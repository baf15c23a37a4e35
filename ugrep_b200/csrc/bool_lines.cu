// bool_lines.cu — Boolean line queries (`ugrep -e A --and -e B`, `A --andnot B`, `--bool`, `--not`, ugx_*_lines_bool):
// from the K terms' matching line records, one term mask per line, the clauses evaluated on it, and one ugx_line per
// selected line in input order.
//
//   bool_mark_kernel   after term j's selection (the matching records of ugx_find_lines), mask[line - 1] |= 1 << j
//                      for each of its records.  A line occurs at most once per term: no atomics.
//   bool_count_kernel  block b counts the selected lines of line block b (BOOL_LINES_PER_BLOCK lines) and, when the
//                      records are wanted, the '\n' bytes of byte region b (BOOL_REGION bytes).  The clauses come by
//                      value in the kernel parameters.
//   tile prefix        launch_tile_prefix over both columns: every line block's first output slot, every region's
//                      first line, and the totals {selected lines, newlines}.
//   bool_index_kernel  region b writes eol[i] = offset of line i's '\n' for each newline in it (and the buffer end for
//                      an unterminated last line), so that every line has its position, M(L) = 0 included.
//   bool_emit_kernel   line block b writes every selected line to its final slot: a ballot orders the lanes, the
//                      block prefix orders the blocks.  No atomics.
#include "scan_kernels.hpp"

namespace ugx {

namespace {

constexpr int BOOL_THREADS = 256;
constexpr uint32_t FULL = 0xffffffffu;

__device__ __forceinline__ bool bool_selected(const BoolQuery& q, uint32_t m)
{
  bool ok = true;
  for (uint32_t c = 0; c < q.nclauses; ++c)
    if (((m & q.pos[c]) | (~m & q.neg[c])) == 0)
    {
      ok = false;
      break;
    }
  return ok != (q.invert != 0);
}

// bit k = byte k of the 16 bytes at buf + c is '\n' (bytes at or past n read as none)
__device__ __forceinline__ uint32_t bool_newlines16(const uint8_t* buf, uint64_t n, uint64_t c)
{
  uint32_t w[4];
  if (c + 16 <= n)
  {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(buf + c));
    w[0] = v.x;
    w[1] = v.y;
    w[2] = v.z;
    w[3] = v.w;
  }
  else
  {
#pragma unroll
    for (int k = 0; k < 4; ++k)
    {
      w[k] = 0;
#pragma unroll
      for (int b = 0; b < 4; ++b)
        if (c + 4 * k + b < n)
          w[k] |= static_cast<uint32_t>(__ldg(buf + c + 4 * k + b)) << (8 * b);
    }
  }
  uint32_t m = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k)
  {
    const uint32_t e = __vcmpeq4(w[k], 0x0a0a0a0au) & 0x80808080u;
    m |= ((e >> 7) | (e >> 14) | (e >> 21) | (e >> 28)) << (4 * k) & (0xfu << (4 * k));
  }
  return m;
}

// exclusive prefix of v over the CTA, and the CTA's total
__device__ __forceinline__ uint32_t block_excl_scan32(uint32_t v, uint32_t* warp_sums, uint32_t* total)
{
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1)
  {
    const uint32_t y = __shfl_up_sync(FULL, x, d);
    if (lane >= static_cast<uint32_t>(d))
      x += y;
  }
  if (lane == 31)
    warp_sums[wid] = x;
  __syncthreads();
  uint32_t before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < BOOL_THREADS / 32; ++w)
  {
    const uint32_t s = warp_sums[w];
    before += w < static_cast<int>(wid) ? s : 0u;
    all += s;
  }
  __syncthreads();
  *total = all;
  return x - v + before;
}

__device__ __forceinline__ uint64_t block_sum64(uint64_t v, uint64_t* sums)
{
#pragma unroll
  for (int d = 16; d > 0; d >>= 1)
    v += __shfl_down_sync(FULL, v, d);
  if ((threadIdx.x & 31) == 0)
    sums[threadIdx.x >> 5] = v;
  __syncthreads();
  uint64_t all = 0;
#pragma unroll
  for (int w = 0; w < BOOL_THREADS / 32; ++w)
    all += sums[w];
  return all;
}

} // namespace

__global__ void __launch_bounds__(BOOL_THREADS)
bool_mark_kernel(const ugx_line* __restrict__ rec, uint64_t nrec, uint32_t* __restrict__ mask, uint32_t bit)
{
  for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * BOOL_THREADS + threadIdx.x; i < nrec;
       i += static_cast<uint64_t>(gridDim.x) * BOOL_THREADS)
    mask[rec[i].line - 1] |= bit;
}

__global__ void __launch_bounds__(BOOL_THREADS)
bool_count_kernel(BoolArgs a, const __grid_constant__ BoolQuery q)
{
  __shared__ uint64_t sums[BOOL_THREADS / 32];
  const uint64_t l0 = static_cast<uint64_t>(blockIdx.x) * BOOL_LINES_PER_BLOCK;
  uint64_t sel = 0;
  for (uint32_t k = threadIdx.x; k < BOOL_LINES_PER_BLOCK && l0 + k < a.nlines; k += BOOL_THREADS)
    sel += bool_selected(q, a.mask[l0 + k]) ? 1u : 0u;
  uint64_t nl = 0;
  if (a.want_index)
  {
    const uint64_t r0 = static_cast<uint64_t>(blockIdx.x) * BOOL_REGION;
    for (uint32_t k = 16 * threadIdx.x; k < BOOL_REGION && r0 + k < a.n; k += 16 * BOOL_THREADS)
      nl += __popc(bool_newlines16(a.buf, a.n, r0 + k));
  }
  sel = block_sum64(sel, sums);
  __syncthreads();
  nl = block_sum64(nl, sums);
  if (threadIdx.x == 0)
  {
    a.blk[blockIdx.x] = sel;
    a.blk[a.nblocks + blockIdx.x] = nl;
  }
}

__global__ void __launch_bounds__(BOOL_THREADS)
bool_index_kernel(BoolArgs a)
{
  __shared__ uint32_t warp_sums[BOOL_THREADS / 32];
  const uint64_t r0 = static_cast<uint64_t>(blockIdx.x) * BOOL_REGION;
  uint64_t at = a.blk[a.nblocks + blockIdx.x]; // lines that end before the region
  for (uint32_t k = 0; k < BOOL_REGION && r0 + k < a.n; k += 16 * BOOL_THREADS)
  {
    const uint64_t c = r0 + k + 16 * threadIdx.x;
    uint32_t m = c < a.n ? bool_newlines16(a.buf, a.n, c) : 0u;
    uint32_t total;
    uint64_t i = at + block_excl_scan32(__popc(m), warp_sums, &total);
    while (m != 0)
    {
      a.eol[i++] = c + (__ffs(m) - 1);
      m &= m - 1;
    }
    at += total;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && __ldg(a.buf + a.n - 1) != '\n')
    a.eol[a.nlines - 1] = a.n;
}

__global__ void __launch_bounds__(BOOL_THREADS)
bool_emit_kernel(BoolArgs a, const __grid_constant__ BoolQuery q)
{
  __shared__ uint32_t warp_sums[BOOL_THREADS / 32];
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t l0 = static_cast<uint64_t>(blockIdx.x) * BOOL_LINES_PER_BLOCK;
  uint64_t at = a.blk[blockIdx.x]; // selected lines before the block
  for (uint32_t k = 0; k < BOOL_LINES_PER_BLOCK && l0 + k < a.nlines; k += BOOL_THREADS)
  {
    const uint64_t i = l0 + k + threadIdx.x;
    const uint32_t m = i < a.nlines ? a.mask[i] : 0u;
    const bool s = i < a.nlines && bool_selected(q, m);
    const uint32_t ballot = __ballot_sync(FULL, s);
    uint32_t total;
    const uint32_t wbase = block_excl_scan32(lane == 0 ? __popc(ballot) : 0u, warp_sums, &total);
    const uint64_t slot = at + __shfl_sync(FULL, wbase, 0) + __popc(ballot & ((1u << lane) - 1u));
    if (s)
    {
      ugx_line r;
      r.line = a.base_line + i + 1;
      r.bol = a.base_offset + (i == 0 ? 0 : a.eol[i - 1] + 1);
      r.eol = a.base_offset + a.eol[i];
      r.offset = r.bol;
      r.len = 0;
      r.cap = m;
      a.out[slot] = r;
    }
    at += total;
  }
}

uint64_t bool_line_blocks(uint64_t nlines) { return (nlines + BOOL_LINES_PER_BLOCK - 1) / BOOL_LINES_PER_BLOCK; }
uint64_t bool_regions(uint64_t n) { return (n + BOOL_REGION - 1) / BOOL_REGION; }

cudaError_t launch_bool_mark(const ugx_line* rec, uint64_t nrec, uint32_t* mask, uint32_t bit, int sm_count,
                             cudaStream_t st)
{
  uint64_t g = (nrec + BOOL_THREADS - 1) / BOOL_THREADS;
  const uint64_t gmax = static_cast<uint64_t>(sm_count) * 16;
  if (g > gmax)
    g = gmax;
  if (g == 0)
    g = 1;
  bool_mark_kernel<<<static_cast<unsigned>(g), BOOL_THREADS, 0, st>>>(rec, nrec, mask, bit);
  return cudaGetLastError();
}

cudaError_t launch_bool_count(const BoolArgs& a, const BoolQuery& q, cudaStream_t st)
{
  bool_count_kernel<<<static_cast<unsigned>(a.nblocks), BOOL_THREADS, 0, st>>>(a, q);
  return cudaGetLastError();
}

cudaError_t launch_bool_index(const BoolArgs& a, cudaStream_t st)
{
  bool_index_kernel<<<static_cast<unsigned>(bool_regions(a.n)), BOOL_THREADS, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_bool_emit(const BoolArgs& a, const BoolQuery& q, cudaStream_t st)
{
  bool_emit_kernel<<<static_cast<unsigned>(bool_line_blocks(a.nlines)), BOOL_THREADS, 0, st>>>(a, q);
  return cudaGetLastError();
}

} // namespace ugx
