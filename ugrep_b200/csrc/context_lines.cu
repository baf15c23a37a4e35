// context_lines.cu — context lines (`ugrep -A NUM -B NUM -C NUM`, ugx_find_context*): from the selected line records
// of ugx_find_lines[_batch], one ugx_line per printed line in input order.  A line is printed when some selected line s
// has s - before <= line <= s + after (GNU grep's rule, which ugrep follows); windows stop at the first and last line
// of their buffer or file.
//
//   context_count_kernel  one thread per selected record, line numbers only.  Record i owns its after-context
//                         L_i+1 .. min(L_i+after, L_{i+1}-1, last) and its before-context
//                         max(L_i-before, L_{i-1}+after+1, 1) .. L_i-1, so every printed line has exactly one owner.
//                         Output: 1 + owned lines, as an exclusive prefix within blocks of CTX_PER_BLOCK records
//                         (pos[]) and the block sums (blk[]).
//   tile prefix           launch_tile_prefix over the block sums: each block's output position, and the total.
//   context_emit_kernel   a warp per 32 records: each lane copies its selected record to its final slot, then the
//                         warp walks out from every record with context, backward from bol - 1 and forward from
//                         eol + 1, 512 bytes a step (16 per lane, a popc scan orders the newlines).  The walk reads
//                         only the text of the printed context lines; no atomics.
//   context_match_kernel  under UGX_LINES_INVERT only: a context line is then a matching line, and a thread per
//                         printed line runs find_in_line on it, as scan_lines_kernel does.  A kernel of its own keeps
//                         the DFA code out of the walk.
#include "block_scan.cuh"
#include "device_pattern.cuh"
#include "line_match.cuh"
#include "line_stage.cuh"
#include "scan_kernels.hpp"

namespace ugx {

namespace {

constexpr int CTX_THREADS = 256;
constexpr uint32_t FULL = 0xffffffffu;

// the file record i belongs to: its records [lo, hi), its bytes, its newlines (one buffer: file 0 is the buffer)
struct CtxFile {
  uint64_t lo, hi;
  uint64_t begin, len;
  uint32_t f;
};

__device__ __forceinline__ CtxFile ctx_file(const ContextArgs& a, uint64_t i)
{
  CtxFile F;
  if (a.fsel == nullptr)
  {
    F.lo = 0;
    F.hi = a.nsel;
    F.begin = 0;
    F.len = a.n;
    F.f = 0;
    return F;
  }
  // the last file whose first record is <= i (empty files share their first record with the next file)
  const uint64_t lo = last_le(a.fsel, 0, a.nfiles, i);
  F.f = static_cast<uint32_t>(lo);
  F.lo = a.fsel[lo];
  F.hi = a.fsel[lo + 1];
  F.begin = a.begins[lo];
  F.len = a.lens[lo];
  return F;
}

// the file's last line number: its newlines, plus one when it does not end in '\n'
__device__ __forceinline__ uint64_t ctx_last_line(const ContextArgs& a, const CtxFile& F)
{
  uint64_t nl = a.nl_total;
  if (a.fsel != nullptr)
  {
    const uint64_t t0 = a.ftile[F.f], t1 = a.ftile[F.f + 1];
    nl = (t1 < a.ntiles ? a.tile_nl[t1] : a.nl_total) - (t0 < a.ntiles ? a.tile_nl[t0] : a.nl_total);
  }
  const bool tail = F.len > 0 && __ldg(a.buf + F.begin + F.len - 1) != '\n';
  return a.base_line + nl + (tail ? 1u : 0u);
}

// the before- and after-context record i owns (saturating: no window arithmetic wraps)
__device__ __forceinline__ void ctx_window(const ContextArgs& a, const CtxFile& F, uint64_t i, uint64_t L, uint64_t& cb,
                                           uint64_t& ca)
{
  uint64_t lim = a.base_line + 1; // first line the before-context may take
  if (i > F.lo)
  {
    const uint64_t P = a.sel[i - 1].line; // < L
    lim = P + (a.after < L - 1 - P ? a.after : L - 1 - P) + 1;
  }
  cb = a.before < L - lim ? a.before : L - lim;
  const uint64_t hi = i + 1 < F.hi ? a.sel[i + 1].line - 1 : ctx_last_line(a, F); // >= L
  ca = a.after < hi - L ? a.after : hi - L;
}

// one context line t[b, e) (e = its '\n', or the end of the file) without a match; under invert it is a matching line
// and context_match_kernel fills in its first match (len = ~0 marks it)
__device__ __forceinline__ void put_context(const ContextArgs& a, uint64_t line, uint64_t b, uint64_t e, uint64_t off,
                                            ugx_line* dst)
{
  ugx_line r;
  r.line = line;
  r.bol = b + off;
  r.eol = e + off;
  r.offset = r.bol;
  r.len = a.invert ? ~0u : 0u;
  r.cap = 0;
  *dst = r;
}

// the k lines after the line whose '\n' is at e: dst[j] = line `line` + 1 + j.  Warp-uniform arguments.
__device__ __forceinline__ void walk_after(const ContextArgs& a, const Text& t, uint64_t e, uint64_t line,
                           uint64_t k, uint64_t off, ugx_line* dst)
{
  const uint32_t lane = threadIdx.x & 31;
  uint64_t bol = e + 1, found = 0; // start of the next line, lines found
  for (uint64_t p = bol & ~15ull; found < k && p < t.end; p += 32 * 16)
  {
    const uint64_t c = p + 16ull * lane;
    uint32_t m = 0;
    if (c < t.end)
    {
      m = newlines16(t.b, t.end, c);
      if (c < bol)
        m &= 0xffffu << (bol - c);
    }
    const uint32_t cnt = __popc(m);
    uint32_t incl = cnt;
    uint64_t mx = m ? c + (31 - __clz(m)) + 1 : 0; // one past the lane's last newline
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
    {
      const uint32_t y = __shfl_up_sync(FULL, incl, d);
      const uint64_t z = __shfl_up_sync(FULL, mx, d);
      if (lane >= static_cast<uint32_t>(d))
      {
        incl += y;
        mx = z > mx ? z : mx;
      }
    }
    uint64_t b = __shfl_up_sync(FULL, mx, 1);
    if (lane == 0 || b == 0)
      b = bol;
    uint64_t j = found + (incl - cnt);
    while (m != 0 && j < k)
    {
      const uint64_t q = c + (__ffs(m) - 1);
      m &= m - 1;
      put_context(a, line + 1 + j, b, q, off, dst + j);
      b = q + 1;
      ++j;
    }
    found += __shfl_sync(FULL, incl, 31);
    const uint64_t top = __shfl_sync(FULL, mx, 31);
    if (top != 0)
      bol = top;
  }
  if (found < k && lane == 0) // the file's last line, without '\n'
    put_context(a, line + 1 + found, bol, t.end, off, dst + found);
}

// the k lines before the line that starts at s + 1 (s its predecessor's '\n'): dst[-1 - j] = line `line` - 1 - j.
__device__ __forceinline__ void walk_before(const ContextArgs& a, const Text& t, uint64_t s, uint64_t line,
                            uint64_t k, uint64_t off, ugx_line* dst)
{
  const uint32_t lane = threadIdx.x & 31;
  uint64_t eol = s, found = 0; // end of the next line (going down), lines found
  // lane l reads the 16 bytes at p - 16 (l + 1): lane 0 the highest
  for (uint64_t p = (s + 15) & ~15ull; found < k && p > 0; p = p > 32 * 16 ? p - 32 * 16 : 0)
  {
    const uint64_t c = p - 16ull * (lane + 1);
    uint32_t m = 0;
    if (p >= 16ull * (lane + 1))
    {
      m = newlines16(t.b, t.end, c);
      if (c + 16 > s)
        m &= (1u << (s - c)) - 1u; // below s only (s - c < 16)
    }
    const uint32_t cnt = __popc(m);
    uint32_t incl = cnt;
    uint64_t mn = m ? c + (__ffs(m) - 1) : ~0ull; // the lane's lowest newline
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
    {
      const uint32_t y = __shfl_up_sync(FULL, incl, d);
      const uint64_t z = __shfl_up_sync(FULL, mn, d);
      if (lane >= static_cast<uint32_t>(d))
      {
        incl += y;
        mn = z < mn ? z : mn;
      }
    }
    uint64_t e = __shfl_up_sync(FULL, mn, 1);
    if (lane == 0 || e == ~0ull)
      e = eol;
    uint64_t j = found + (incl - cnt);
    while (m != 0 && j < k)
    {
      const uint64_t q = c + (31 - __clz(m));
      m &= ~(1u << (q - c));
      put_context(a, line - 1 - j, q + 1, e, off, dst - 1 - j);
      e = q;
      ++j;
    }
    found += __shfl_sync(FULL, incl, 31);
    const uint64_t low = __shfl_sync(FULL, mn, 31);
    if (low != ~0ull)
      eol = low;
  }
  if (found < k && lane == 0) // the file's first line
    put_context(a, line - 1 - found, 0, eol, off, dst - 1 - found);
}

} // namespace

__global__ void __launch_bounds__(CTX_THREADS)
context_count_kernel(ContextArgs a)
{
  __shared__ uint64_t warp_sums[33];
  const uint64_t b0 = static_cast<uint64_t>(blockIdx.x) * CTX_PER_BLOCK;
  uint64_t run = 0;
  for (uint32_t k = 0; k < CTX_PER_BLOCK && b0 + k < a.nsel; k += CTX_THREADS)
  {
    const uint64_t i = b0 + k + threadIdx.x;
    uint64_t c = 0;
    if (i < a.nsel)
    {
      const CtxFile F = ctx_file(a, i);
      uint64_t cb, ca;
      ctx_window(a, F, i, a.sel[i].line, cb, ca);
      c = 1 + cb + ca;
    }
    uint64_t tot;
    const uint64_t ex = block_excl_scan(c, warp_sums, &tot);
    if (i < a.nsel)
      a.pos[i] = run + ex;
    run += tot;
  }
  if (threadIdx.x == 0)
  {
    a.blk[blockIdx.x] = run;
    a.blk[gridDim.x + blockIdx.x] = 0; // launch_tile_prefix's second column
  }
}

__global__ void __launch_bounds__(CTX_THREADS)
context_emit_kernel(ContextArgs a)
{
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * CTX_THREADS + threadIdx.x) / 32;
  const uint64_t nwarps = static_cast<uint64_t>(gridDim.x) * (CTX_THREADS / 32);
  for (uint64_t w0 = warp * 32; w0 < a.nsel; w0 += nwarps * 32)
  {
    const uint64_t i = w0 + lane;
    uint64_t cb = 0, ca = 0, at = 0, line = 0, bol = 0, eol = 0, begin = 0, len = 0;
    if (i < a.nsel)
    {
      const CtxFile F = ctx_file(a, i);
      const ugx_line r = a.sel[i];
      ctx_window(a, F, i, r.line, cb, ca);
      at = a.blk[i / CTX_PER_BLOCK] + a.pos[i] + cb;
      a.out[at] = r;
      line = r.line;
      bol = r.bol - a.base_offset;
      eol = r.eol - a.base_offset;
      begin = F.begin;
      len = F.len;
    }
    uint32_t todo = __ballot_sync(FULL, cb + ca != 0);
    while (todo != 0)
    {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint64_t kb = __shfl_sync(FULL, cb, src), ka = __shfl_sync(FULL, ca, src);
      const uint64_t o = __shfl_sync(FULL, at, src), L = __shfl_sync(FULL, line, src);
      const Text t{a.buf + __shfl_sync(FULL, begin, src), __shfl_sync(FULL, len, src)};
      const uint64_t b = __shfl_sync(FULL, bol, src), e = __shfl_sync(FULL, eol, src);
      if (kb != 0)
        walk_before(a, t, b - 1, L, kb, a.base_offset, a.out + o);
      if (ka != 0)
        walk_after(a, t, e, L, ka, a.base_offset, a.out + o + 1);
    }
  }
  // a batch: every file's first printed line (the position of its first selected record, or of the next file's)
  if (a.fout != nullptr)
    for (uint64_t f = static_cast<uint64_t>(blockIdx.x) * CTX_THREADS + threadIdx.x; f <= a.nfiles;
         f += static_cast<uint64_t>(gridDim.x) * CTX_THREADS)
    {
      const uint64_t r = a.fsel[f];
      a.fout[f] = r < a.nsel ? a.blk[r / CTX_PER_BLOCK] + a.pos[r] : a.nout;
    }
}

// under invert: the first match of every context line (a matching line), as scan_lines_kernel finds it
template <bool HAS_META>
__global__ void __launch_bounds__(CTX_THREADS, 4)
context_match_kernel(const __grid_constant__ DevPattern P, ContextArgs a)
{
  Tables T;
  T.cls = P.cls;
  T.next = P.next;
  T.pred = P.pred;
  T.tap = P.tap;
  const CandMap cm{nullptr, 0, 0};
  for (uint64_t j = static_cast<uint64_t>(blockIdx.x) * CTX_THREADS + threadIdx.x; j < a.nout;
       j += static_cast<uint64_t>(gridDim.x) * CTX_THREADS)
  {
    if (a.out[j].len != ~0u)
      continue;
    uint64_t begin = 0, len = a.n;
    if (a.fout != nullptr)
    {
      const uint64_t lo = last_le(a.fout, 0, a.nfiles, j);
      begin = a.begins[lo];
      len = a.lens[lo];
    }
    const Text t{a.buf + begin, len};
    ugx_line r = a.out[j];
    const uint64_t b = r.bol - a.base_offset, e = r.eol - a.base_offset;
    Cursor m;
    set_current(t, m, b);
    const uint32_t cap = find_in_line<HAS_META>(t, P, T, cm, m, e < len ? e : len - 1);
    r.offset = cap != 0 ? m.txt + a.base_offset : r.bol;
    r.len = cap != 0 ? m.len : 0u;
    r.cap = cap;
    a.out[j] = r;
  }
}

uint64_t context_blocks(uint64_t nsel) { return (nsel + CTX_PER_BLOCK - 1) / CTX_PER_BLOCK; }

cudaError_t launch_context_count(const ContextArgs& a, cudaStream_t st)
{
  context_count_kernel<<<static_cast<unsigned>(context_blocks(a.nsel)), CTX_THREADS, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_context_emit(const ContextArgs& a, int sm_count, cudaStream_t st)
{
  const unsigned g = capped_grid(a.nsel, CTX_THREADS, sm_count, 8); // a warp per 32 records
  context_emit_kernel<<<g, CTX_THREADS, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_context_match(const DevPattern& P, const ContextArgs& a, int sm_count, cudaStream_t st)
{
  const unsigned g = capped_grid(a.nout, CTX_THREADS, sm_count, 8);
  if (P.has_meta)
    context_match_kernel<true><<<g, CTX_THREADS, 0, st>>>(P, a);
  else
    context_match_kernel<false><<<g, CTX_THREADS, 0, st>>>(P, a);
  return cudaGetLastError();
}

} // namespace ugx
