// bool_lines.cu — Boolean line queries (`ugrep -e A --and -e B`, `A --andnot B`, `--bool`, `--not`, ugx_*_lines_bool,
// ugx_*_lines_bool_batch): from the K terms' matching line records, one term mask per line, the clauses evaluated on it,
// and one ugx_line per selected line in input order.
//
// One buffer:
//   bool_mark_kernel   after term j's selection (the matching records of ugx_find_lines), mask[line - 1] |= 1 << j
//                      for each of its records.  A line occurs at most once per term: no atomics.
//   bool_count_kernel  block b counts the selected lines of line block b (BOOL_LINES_PER_BLOCK lines) and, when the
//                      records are wanted, the '\n' bytes of byte region b (BOOL_REGION bytes) and the emit pass's
//                      one-file line table lb = {0, nlines}.  The clauses come by value in the kernel parameters.
//   tile prefix        launch_tile_prefix over both columns: every line block's first output slot, every region's
//                      first line, and the totals {selected lines, newlines}.
//   bool_index_kernel  region b writes eol[i] = offset of line i's '\n' for each newline in it (and the buffer end for
//                      an unterminated last line), so that every line has its position, M(L) = 0 included.
//
// Many files: the batch's lines are numbered across the files, file f owning the global lines [lb[f], lb[f + 1]), an
// empty file none.
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
//
// Both:
//   bool_batch_emit_kernel   line block b writes every selected line to its final slot, in its file's numbering plus
//                            the call's bases: a ballot orders the lanes, the block prefix orders the blocks.  No atomics.
//
// Mark and count have a kernel for each form.  The records of one buffer come with no tile table, and a one-tile table
// would put every record on one warp.  The count of one buffer also counts the newlines per region that its index
// pass needs; the count of a batch makes per-file counts and takes the newline positions from the selection's tile
// prefix.
#include "block_scan.cuh"
#include "line_stage.cuh"
#include "scan_kernels.hpp"

namespace ugx {

namespace {

constexpr int BOOL_THREADS = 256;
constexpr uint32_t FULL = 0xffffffffu;
constexpr uint32_t NO_FILE = 0xffffffffu;

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
  return static_cast<uint32_t>(last_le(lb, l, h < nfiles ? h : nfiles, i));
}

// eol[at + r] = offset of the r-th '\n' of text[c0, c1), 16 bytes a thread; when c1 is the end of the text and its last
// line has no '\n', eol[*lines_end - 1] = len (lines_end: the text's lb[f + 1])
__device__ __forceinline__ void index_lines(const uint8_t* text, uint64_t len, uint64_t c0, uint64_t c1, uint64_t at,
                                            const uint64_t* lines_end, uint64_t* eol, uint32_t* warp_sums)
{
  for (uint64_t k = c0; k < c1; k += 16 * BOOL_THREADS)
  {
    const uint64_t c = k + 16 * threadIdx.x;
    uint32_t m = c < c1 ? newlines16(text, c1, c) : 0u;
    uint32_t total;
    uint64_t i = at + block_excl_scan(static_cast<uint32_t>(__popc(m)), warp_sums, &total);
    while (m != 0)
    {
      eol[i++] = c + (__ffs(m) - 1);
      m &= m - 1;
    }
    at += total;
  }
  if (threadIdx.x == 0 && c1 == len && __ldg(text + len - 1) != '\n')
    eol[*lines_end - 1] = len;
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
      nl += __popc(newlines16(a.buf, a.n, r0 + k));
  }
  sel = block_sum<BOOL_THREADS>(sel, sums);
  __syncthreads();
  nl = block_sum<BOOL_THREADS>(nl, sums);
  if (threadIdx.x == 0)
  {
    a.blk[blockIdx.x] = sel;
    a.blk[a.nblocks + blockIdx.x] = nl;
    if (blockIdx.x == 0 && a.want_index)
    {
      a.lb[0] = 0;
      a.lb[1] = a.nlines;
    }
  }
}

__global__ void __launch_bounds__(BOOL_THREADS)
bool_index_kernel(BoolArgs a)
{
  __shared__ uint32_t warp_sums[33];
  const uint64_t r0 = static_cast<uint64_t>(blockIdx.x) * BOOL_REGION;
  const uint64_t r1 = r0 + BOOL_REGION < a.n ? r0 + BOOL_REGION : a.n;
  const uint64_t at = a.blk[a.nblocks + blockIdx.x]; // lines that end before the region
  index_lines(a.buf, a.n, r0, r1, at, a.lb + 1, a.eol, warp_sums);
}

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
bool_batch_count_kernel(BoolArgs a, const __grid_constant__ BoolQuery q)
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
  const uint64_t all = block_sum<BOOL_THREADS>(lane == 0 ? wsel : 0, sums); // wsel is the same in every lane
  if (threadIdx.x == 0)
  {
    a.blk[blockIdx.x] = all;
    a.blk[a.nblocks + blockIdx.x] = 0;
  }
}

__global__ void __launch_bounds__(BOOL_THREADS)
bool_batch_index_kernel(BoolArgs a)
{
  __shared__ uint32_t warp_sums[33];
  const uint64_t g = blockIdx.x;
  const uint32_t f = a.files.tile_file[g], ti = a.files.tile_index[g];
  const uint64_t len = a.files.lens[f];
  const uint64_t t0 = static_cast<uint64_t>(ti) * SCAN_TILE;
  const uint64_t t1 = t0 + SCAN_TILE < len ? t0 + SCAN_TILE : len;
  // lines of the batch before the tile: the file's first line, and the file's newlines before the tile
  const uint64_t at = a.lb[f] + a.tile_nl[g] - a.tile_nl[g - ti];
  index_lines(a.buf + a.files.begins[f], len, t0, t1, at, a.lb + f + 1, a.eol, warp_sums);
}

__global__ void __launch_bounds__(BOOL_THREADS)
bool_batch_emit_kernel(BoolArgs a, const __grid_constant__ BoolQuery q)
{
  __shared__ uint32_t warp_sums[33];
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
    const uint32_t wbase = block_excl_scan(lane == 0 ? static_cast<uint32_t>(__popc(ballot)) : 0u, warp_sums, &total);
    const uint64_t slot = at + __shfl_sync(FULL, wbase, 0) + __popc(ballot & ((1u << lane) - 1u));
    if (s)
    {
      const uint32_t f = bool_file_of(a.lb, a.nfiles, hint, i);
      hint = f;
      const uint64_t first = a.lb[f];
      ugx_line r;
      r.line = a.base_line + i - first + 1;
      r.bol = a.base_offset + (i == first ? 0 : a.eol[i - 1] + 1);
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
  bool_mark_kernel<<<capped_grid(nrec, BOOL_THREADS, sm_count, 16), BOOL_THREADS, 0, st>>>(rec, nrec, mask, bit);
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
  bool_batch_mark_kernel<<<capped_grid(b.ntiles, BOOL_THREADS / 32, sm_count, 16), BOOL_THREADS, 0, st>>>(
      rec, nrec, tile_rec, b.tile_file, b.ntiles, lb, mask, bit);
  return cudaGetLastError();
}

cudaError_t launch_bool_batch_count(const BoolArgs& a, const BoolQuery& q, cudaStream_t st)
{
  bool_batch_count_kernel<<<static_cast<unsigned>(a.nblocks), BOOL_THREADS, 0, st>>>(a, q);
  return cudaGetLastError();
}

cudaError_t launch_bool_batch_index(const BoolArgs& a, cudaStream_t st)
{
  bool_batch_index_kernel<<<static_cast<unsigned>(a.files.ntiles), BOOL_THREADS, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_bool_batch_emit(const BoolArgs& a, const BoolQuery& q, cudaStream_t st)
{
  bool_batch_emit_kernel<<<static_cast<unsigned>(bool_line_blocks(a.nlines)), BOOL_THREADS, 0, st>>>(a, q);
  return cudaGetLastError();
}

} // namespace ugx
