// batch_records.cu — match and line records of many files in one launch sequence (ugx_find_all_batch,
// ugx_find_lines_batch): the two-pass form of scan_batch_kernel (batch_kernel.cu) over the same tile table, 16 KiB
// tiles with a Text{buf + begin, len} per tile, so every file keeps its own end of buffer.
//
//   count pass   the records every 64-byte strip owns -> strip_counts, {records, newlines} of every batch tile,
//                and the per-file record counts (one atomic per tile)
//   tile prefix  launch_tile_prefix over the batch tiles: they are ordered by file, then by offset, so the exclusive
//                prefix is each tile's output position, and newlines before the file's first tile give line numbers
//   emit pass    the same strip-owner walk; every record goes to its final slot without atomics
//
// A translation unit of its own, so that the counting kernel of batch_kernel.cu keeps its code generation.
#include "block_scan.cuh"
#include "device_pattern.cuh"
#include "line_match.cuh"
#include "ptx.cuh"
#include "scan_kernels.hpp"
#include "tile_phase_a.cuh"

namespace ugx {

// LINES: one ugx_line per line whose first find_in_line result is a match, or with r.lflags & UGX_LINES_INVERT per line
// where it is none (scan_lines_kernel's LINES form); otherwise one ugx_match per find_in_line result (its MODE 1 record
// pass).  r.lflags & SCAN_LINES_NEVER: the pattern admits no candidate, no line is searched.
template <bool EMIT, bool HAS_META, bool LINES>
__global__ void __launch_bounds__(SCAN_THREADS, 4)
scan_batch_records_kernel(const __grid_constant__ DevPattern P, const uint8_t* __restrict__ buf, BatchArgs a,
                          BatchRecordArgs r)
{
  constexpr uint32_t TILE = SCAN_TILE;
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ uint32_t warp_sums[33];
  __shared__ uint32_t red_m[SCAN_THREADS / 32], red_n[SCAN_THREADS / 32];
  uint8_t* s_cls = smem;
  uint8_t* s_pred = smem + 256;
  uint8_t* s_tap = s_pred + UGX_HASH;
  uint32_t* s_cand = reinterpret_cast<uint32_t*>(s_tap + UGX_BTAP);
  uint32_t* s_nl = s_cand + TILE / 32;
  uint16_t* s_next = reinterpret_cast<uint16_t*>(s_nl + TILE / 32);
  stage_tables_bulk(&s_bar, s_cls, P.cls, s_pred, P.pred, s_tap, P.tap, s_next, P.next,
                    a.stage_table ? ((P.table_bytes + 15) / 16) * 16 : 0);
  __syncthreads();
  Tables T;
  T.cls = s_cls;
  T.pred = s_pred;
  T.tap = s_tap;
  T.next = a.stage_table ? s_next : P.next;
  const bool never = (r.lflags & SCAN_LINES_NEVER) != 0;
  const bool inv = (r.lflags & UGX_LINES_INVERT) != 0;
  for (uint64_t g = blockIdx.x; g < a.ntiles; g += gridDim.x)
  {
    // emit pass: a tile without records has nothing to write (the same value for the whole block)
    if (EMIT && (g + 1 < a.ntiles ? r.tile_matches[g + 1] : r.out_cap) == r.tile_matches[g])
      continue;
    const uint32_t f = a.tile_file[g];
    const uint32_t ti = a.tile_index[g];
    const uint64_t begin = a.begins[f], len = a.lens[f];
    const uint64_t tile_base = static_cast<uint64_t>(ti) * TILE; // within the file
    const Text t{buf + begin, len};
    const uint64_t s0 = tile_base + static_cast<uint64_t>(threadIdx.x) * SCAN_STRIP;
    tile_phase_a<TILE / 16 / SCAN_THREADS>(t, P, T, tile_base, reinterpret_cast<uint16_t*>(s_cand),
                                           reinterpret_cast<uint16_t*>(s_nl));
    __syncthreads();
    const CandMap cm{s_cand, tile_base, TILE};
    // phase A leaves no newline past the end of the file: the padding between files is never counted
    const uint64_t nl = (static_cast<uint64_t>(s_nl[2 * threadIdx.x + 1]) << 32) | s_nl[2 * threadIdx.x];
    const uint32_t my_nl = __popcll(nl);
    uint64_t starts = nl << 1;
    if (s0 < len && (s0 == 0 || t.raw(s0 - 1) == '\n'))
      starts |= 1ull;
    if (s0 >= len)
      starts = 0;
    else if (len - s0 < 64)
      starts &= (1ull << (len - s0)) - 1;
    if (!LINES && never)
      starts = 0;

    uint64_t out_pos = 0, line_no = 0;
    if (EMIT)
    {
      uint32_t tot;
      out_pos = r.tile_matches[g] + block_excl_scan(r.strip_counts[g * SCAN_THREADS + threadIdx.x], warp_sums, &tot);
      // line numbers restart in every file: newlines before this tile, less those before the file's first tile
      line_no = 1 + r.tile_newlines[g] - r.tile_newlines[g - ti] + block_excl_scan(my_nl, warp_sums, &tot);
    }

    uint32_t strip_total = 0;
    uint64_t rest = starts;
    while (rest != 0)
    {
      const uint32_t bit = __ffsll(static_cast<long long>(rest)) - 1;
      rest &= rest - 1;
      const uint64_t L = s0 + bit;
      // end of the line: its '\n', or the last byte of the file
      uint64_t last;
      const uint64_t after = nl >> bit;
      if (after != 0)
        last = L + (__ffsll(static_cast<long long>(after)) - 1);
      else
      {
        uint64_t p = s0 + SCAN_STRIP;
        while (p < len && t.raw(p) != '\n')
          ++p;
        last = p < len ? p : len - 1;
      }
      uint64_t this_line = 0;
      if (EMIT)
        this_line = line_no + __popcll(nl & ((1ull << bit) - 1));
      Cursor m;
      set_current(t, m, L);
      if (LINES)
      {
        // the `ugrep -c` loop's view of the line: its first find, then on to the next line
        const uint32_t cap = never ? 0u : find_in_line<HAS_META>(t, P, T, cm, m, last);
        if ((cap != 0) != inv)
        {
          if (EMIT)
          {
            const uint64_t idx = out_pos + strip_total;
            if (idx < r.out_cap)
            {
              ugx_line rec;
              rec.line = this_line;
              rec.bol = L;
              rec.eol = t.raw(last) == '\n' ? last : len;
              rec.offset = inv ? L : m.txt;
              rec.len = inv ? 0u : m.len;
              rec.cap = cap;
              r.lout[idx] = rec;
            }
          }
          ++strip_total;
        }
      }
      else
      {
        // every find_in_line result on the line
        for (;;)
        {
          const uint32_t cap = find_in_line<HAS_META>(t, P, T, cm, m, last);
          if (cap == 0)
            break;
          if (EMIT)
          {
            const uint64_t idx = out_pos + strip_total;
            if (idx < r.out_cap)
            {
              ugx_match rec;
              rec.line = this_line;
              rec.offset = m.txt;
              rec.len = m.len;
              rec.cap = cap;
              r.out[idx] = rec;
            }
          }
          ++strip_total;
        }
      }
    }

    if (!EMIT)
    {
      r.strip_counts[g * SCAN_THREADS + threadIdx.x] = strip_total;
      uint32_t tm = strip_total, tn = my_nl;
#pragma unroll
      for (int d = 16; d > 0; d >>= 1)
      {
        tm += __shfl_down_sync(0xffffffffu, tm, d);
        tn += __shfl_down_sync(0xffffffffu, tn, d);
      }
      if ((threadIdx.x & 31) == 0)
      {
        red_m[threadIdx.x >> 5] = tm;
        red_n[threadIdx.x >> 5] = tn;
      }
      __syncthreads();
      if (threadIdx.x == 0)
      {
        unsigned long long sm = 0, sn = 0;
        for (uint32_t w = 0; w < SCAN_THREADS / 32; ++w)
        {
          sm += red_m[w];
          sn += red_n[w];
        }
        r.tile_matches[g] = sm;
        r.tile_newlines[g] = sn;
        if (sm != 0)
          atomicAdd(a.counts + f, sm);
      }
    }
    __syncthreads(); // the bitmaps are rewritten by the next tile
  }
}

cudaError_t launch_scan_batch_records(const DevPattern& P, const uint8_t* buf, BatchArgs a, const BatchRecordArgs& r,
                                      bool lines, bool emit, int sm_count, cudaStream_t st)
{
  // the shared-memory budget and the grid of launch_scan_batch
  const bool stage = P.has_meta == 0 && P.table_bytes <= SCAN_MAX_SMEM_TABLE;
  const size_t smem = 256 + UGX_HASH + UGX_BTAP + 2 * (SCAN_TILE / 8) + (stage ? ((P.table_bytes + 15) / 16) * 16 : 0);
  a.stage_table = stage ? 1u : 0u;
  int per_sm = static_cast<int>((220 * 1024) / (smem + 1024));
  if (per_sm > 8)
    per_sm = 8;
  if (per_sm < 1)
    per_sm = 1;
  uint64_t g = static_cast<uint64_t>(sm_count) * per_sm;
  if (g > a.ntiles)
    g = a.ntiles;
  if (g == 0)
    g = 1;
#define UGX_BATCH_REC_GO(EMIT, META, LINES)                                                                 \
  do                                                                                                        \
  {                                                                                                         \
    auto kern = scan_batch_records_kernel<EMIT, META, LINES>;                                               \
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, UGX_MAX_DYN_SMEM); \
    if (e != cudaSuccess)                                                                                   \
      return e;                                                                                             \
    kern<<<static_cast<int>(g), SCAN_THREADS, smem, st>>>(P, buf, a, r);                                    \
    return cudaGetLastError();                                                                              \
  } while (0)
#define UGX_BATCH_REC_META(EMIT, LINES) \
  do                                    \
  {                                     \
    if (P.has_meta)                     \
      UGX_BATCH_REC_GO(EMIT, true, LINES); \
    UGX_BATCH_REC_GO(EMIT, false, LINES); \
  } while (0)
  if (lines)
  {
    if (emit)
      UGX_BATCH_REC_META(true, true);
    UGX_BATCH_REC_META(false, true);
  }
  if (emit)
    UGX_BATCH_REC_META(true, false);
  UGX_BATCH_REC_META(false, false);
#undef UGX_BATCH_REC_META
#undef UGX_BATCH_REC_GO
}

} // namespace ugx
