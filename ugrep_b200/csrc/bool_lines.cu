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

// ---- many files (ugx_*_lines_bool_batch) ----
// The batch's lines are numbered across the files: file f owns the global lines [lb[f], lb[f + 1]), an empty file none.
//
//   bool_batch_lines_kernel  the last batch tile of every file writes the file's lines (its newlines, from the tile
//                            newline prefix a term's count pass left, + 1 for an unterminated last line) and newlines;
//                            launch_tile_prefix turns the columns into lb[] and the batch's line count
//   bool_batch_mark_kernel   after term j's selection: one warp per batch tile ORs bit j into the mask of every record
//                            the tile owns (the records of tile g are [tile_rec[g], tile_rec[g + 1]), its file is
//                            tile_file[g]).  A line occurs at most once per term: no atomics.
//   bool_batch_count_kernel  block b: the selected lines of global line block b, and every file's selected lines, one
//                            atomic per warp and file run
//   bool_batch_index_kernel  one block per batch tile: eol[lb[f] + rank] = offset within the file of every '\n' of
//                            the tile, and the file's length for an unterminated last line.  Reads stay in the file.
//   bool_batch_emit_kernel   bool_emit_kernel over the global lines, each record in its file's numbering

namespace {

constexpr uint32_t NO_FILE = 0xffffffffu;

// the last file f >= lo with lb[f] <= i, given lb[lo] <= i < lb[nfiles]: a gallop from lo, then a bisection.  Empty
// files (lb[f] == lb[f + 1]) are passed over.
__device__ __forceinline__ uint32_t bool_file_of(const uint64_t* lb, uint64_t nfiles, uint32_t lo, uint64_t i)
{
  uint64_t l = lo, h = lo, step = 1;
  for (;;)
  {
    h = l + step;
    if (h >= nfiles || __ldg(lb + h) > i)
      break;
    l = h;
    step *= 2;
  }
  if (h > nfiles)
    h = nfiles;
  while (h - l > 1)
  {
    const uint64_t mid = l + (h - l) / 2;
    if (__ldg(lb + mid) <= i)
      l = mid;
    else
      h = mid;
  }
  return static_cast<uint32_t>(l);
}

} // namespace

__global__ void __launch_bounds__(BOOL_THREADS)
bool_batch_lines_kernel(const uint8_t* __restrict__ buf, BatchArgs b, const uint64_t* __restrict__ tile_nl,
                        const unsigned long long* __restrict__ nl_total, uint64_t* __restrict__ flines,
                        uint64_t* __restrict__ fnl)
{
  const uint64_t g = static_cast<uint64_t>(blockIdx.x) * BOOL_THREADS + threadIdx.x;
  if (g >= b.ntiles)
    return;
  const uint32_t f = b.tile_file[g];
  if (g + 1 < b.ntiles && b.tile_file[g + 1] == f)
    return; // not the file's last tile
  const uint64_t end = g + 1 < b.ntiles ? tile_nl[g + 1] : *nl_total;
  const uint64_t nl = end - tile_nl[g - b.tile_index[g]];
  const uint64_t len = b.lens[f];
  fnl[f] = nl;
  flines[f] = nl + (__ldg(buf + b.begins[f] + len - 1) != '\n' ? 1u : 0u);
}

__global__ void __launch_bounds__(BOOL_THREADS)
bool_batch_mark_kernel(const ugx_line* __restrict__ rec, uint64_t nrec, const uint64_t* __restrict__ tile_rec,
                       const uint32_t* __restrict__ tile_file, uint64_t ntiles, const uint64_t* __restrict__ lb,
                       uint32_t* __restrict__ mask, uint32_t bit)
{
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warps = static_cast<uint64_t>(gridDim.x) * (BOOL_THREADS / 32);
  for (uint64_t g = static_cast<uint64_t>(blockIdx.x) * (BOOL_THREADS / 32) + (threadIdx.x >> 5); g < ntiles; g += warps)
  {
    const uint64_t hi = g + 1 < ntiles ? tile_rec[g + 1] : nrec;
    const uint64_t first = lb[tile_file[g]]; // global index of the file's line 1
    for (uint64_t r = tile_rec[g] + lane; r < hi; r += 32)
      mask[first + rec[r].line - 1] |= bit;
  }
}

__global__ void __launch_bounds__(BOOL_THREADS)
bool_batch_count_kernel(BoolBatchArgs a, const __grid_constant__ BoolQuery q)
{
  __shared__ uint32_t s_first;
  __shared__ uint64_t sums[BOOL_THREADS / 32];
  constexpr uint32_t PER_WARP = BOOL_LINES_PER_BLOCK / (BOOL_THREADS / 32);
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint64_t l0 = static_cast<uint64_t>(blockIdx.x) * BOOL_LINES_PER_BLOCK;
  if (threadIdx.x == 0)
    s_first = bool_file_of(a.lb, a.nfiles, 0, l0);
  __syncthreads();
  uint32_t hint = s_first;
  // the warp's lines [w0, w0 + PER_WARP), 32 at a time; the file of the last selected line carries over to the next
  // step, every other file's selected lines of a step go out in one atomic
  const uint64_t w0 = l0 + static_cast<uint64_t>(wid) * PER_WARP;
  uint32_t cur_f = NO_FILE, cur = 0;
  uint64_t wsel = 0;
  for (uint32_t k = 0; k < PER_WARP && w0 + k < a.nlines; k += 32)
  {
    const uint64_t i = w0 + k + lane;
    const bool s = i < a.nlines && bool_selected(q, a.mask[i]);
    const uint32_t any = __ballot_sync(FULL, s);
    if (any == 0)
      continue;
    wsel += __popc(any);
    uint32_t f = NO_FILE;
    if (s)
    {
      f = bool_file_of(a.lb, a.nfiles, hint, i);
      hint = f;
    }
    const uint32_t last = __reduce_max_sync(FULL, s ? f : 0u);
    const uint32_t grp = __match_any_sync(FULL, f);
    if (s && f != last && (grp & ((1u << lane) - 1u)) == 0)
      atomicAdd(a.fsel + f, static_cast<unsigned long long>(__popc(grp)));
    const uint32_t n_last = __popc(__ballot_sync(FULL, s && f == last));
    if (last == cur_f)
      cur += n_last;
    else
    {
      if (lane == 0 && cur != 0)
        atomicAdd(a.fsel + cur_f, static_cast<unsigned long long>(cur));
      cur_f = last;
      cur = n_last;
    }
  }
  if (lane == 0 && cur != 0)
    atomicAdd(a.fsel + cur_f, static_cast<unsigned long long>(cur));
  if (lane == 0)
    sums[wid] = wsel;
  __syncthreads();
  if (threadIdx.x == 0)
  {
    uint64_t all = 0;
#pragma unroll
    for (int w = 0; w < BOOL_THREADS / 32; ++w)
      all += sums[w];
    a.blk[blockIdx.x] = all;
    a.blk[a.nblocks + blockIdx.x] = 0;
  }
}

__global__ void __launch_bounds__(BOOL_THREADS)
bool_batch_index_kernel(BoolBatchArgs a)
{
  __shared__ uint32_t warp_sums[BOOL_THREADS / 32];
  const uint64_t g = blockIdx.x;
  const uint32_t f = a.files.tile_file[g], ti = a.files.tile_index[g];
  const uint8_t* text = a.buf + a.files.begins[f];
  const uint64_t len = a.files.lens[f];
  const uint64_t t0 = static_cast<uint64_t>(ti) * SCAN_TILE;
  const uint64_t t1 = t0 + SCAN_TILE < len ? t0 + SCAN_TILE : len;
  // lines of the batch before the tile: the file's first line, and the file's newlines before the tile
  uint64_t at = a.lb[f] + a.tile_nl[g] - a.tile_nl[g - ti];
  for (uint64_t k = t0; k < t1; k += 16 * BOOL_THREADS)
  {
    const uint64_t c = k + 16 * threadIdx.x;
    uint32_t m = c < t1 ? bool_newlines16(text, t1, c) : 0u;
    uint32_t total;
    uint64_t i = at + block_excl_scan32(__popc(m), warp_sums, &total);
    while (m != 0)
    {
      a.eol[i++] = c + (__ffs(m) - 1);
      m &= m - 1;
    }
    at += total;
  }
  if (threadIdx.x == 0 && t1 == len && __ldg(text + len - 1) != '\n')
    a.eol[a.lb[f + 1] - 1] = len;
}

__global__ void __launch_bounds__(BOOL_THREADS)
bool_batch_emit_kernel(BoolBatchArgs a, const __grid_constant__ BoolQuery q)
{
  __shared__ uint32_t warp_sums[BOOL_THREADS / 32];
  __shared__ uint32_t s_first;
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t l0 = static_cast<uint64_t>(blockIdx.x) * BOOL_LINES_PER_BLOCK;
  if (threadIdx.x == 0)
    s_first = bool_file_of(a.lb, a.nfiles, 0, l0);
  __syncthreads();
  uint32_t hint = s_first;
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
      const uint32_t f = bool_file_of(a.lb, a.nfiles, hint, i);
      hint = f;
      const uint64_t first = a.lb[f];
      ugx_line r;
      r.line = i - first + 1;
      r.bol = i == first ? 0 : a.eol[i - 1] + 1;
      r.eol = a.eol[i];
      r.offset = r.bol;
      r.len = 0;
      r.cap = m;
      a.out[slot] = r;
    }
    at += total;
  }
}

cudaError_t launch_bool_batch_lines(const uint8_t* buf, const BatchArgs& b, const uint64_t* tile_nl,
                                    const unsigned long long* nl_total, uint64_t* flines, uint64_t* fnl, cudaStream_t st)
{
  const uint64_t g = (b.ntiles + BOOL_THREADS - 1) / BOOL_THREADS;
  bool_batch_lines_kernel<<<static_cast<unsigned>(g), BOOL_THREADS, 0, st>>>(buf, b, tile_nl, nl_total, flines, fnl);
  return cudaGetLastError();
}

cudaError_t launch_bool_batch_mark(const ugx_line* rec, uint64_t nrec, const uint64_t* tile_rec, const BatchArgs& b,
                                   const uint64_t* lb, uint32_t* mask, uint32_t bit, int sm_count, cudaStream_t st)
{
  uint64_t g = (b.ntiles + BOOL_THREADS / 32 - 1) / (BOOL_THREADS / 32);
  const uint64_t gmax = static_cast<uint64_t>(sm_count) * 16;
  if (g > gmax)
    g = gmax;
  bool_batch_mark_kernel<<<static_cast<unsigned>(g), BOOL_THREADS, 0, st>>>(rec, nrec, tile_rec, b.tile_file, b.ntiles,
                                                                            lb, mask, bit);
  return cudaGetLastError();
}

cudaError_t launch_bool_batch_count(const BoolBatchArgs& a, const BoolQuery& q, cudaStream_t st)
{
  bool_batch_count_kernel<<<static_cast<unsigned>(a.nblocks), BOOL_THREADS, 0, st>>>(a, q);
  return cudaGetLastError();
}

cudaError_t launch_bool_batch_index(const BoolBatchArgs& a, cudaStream_t st)
{
  bool_batch_index_kernel<<<static_cast<unsigned>(a.files.ntiles), BOOL_THREADS, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_bool_batch_emit(const BoolBatchArgs& a, const BoolQuery& q, cudaStream_t st)
{
  bool_batch_emit_kernel<<<static_cast<unsigned>(a.nblocks), BOOL_THREADS, 0, st>>>(a, q);
  return cudaGetLastError();
}

} // namespace ugx
