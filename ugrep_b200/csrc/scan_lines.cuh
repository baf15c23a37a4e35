// scan_lines.cuh — scan_lines_kernel, the generic exact line scan (see scan_kernels.cu), and the pieces of its
// launchers.  A header so that the line-record instantiations (line_records.cu) compile in a translation unit of
// their own: the counting and match-record kernels of scan_kernels.cu keep their code generation.
#pragma once

#include "device_pattern.cuh"
#include "ptx.cuh"
#include "line_match.cuh"
#include "scan_kernels.hpp"
#include "tile_phase_a.cuh"
#include "block_scan.cuh"

namespace ugx {


// MODE 0: count matching lines (ugrep -c), 1: count matches (ugrep -c -o) / emit records (ugrep -o)
// LINES (with MODE 0, strip-owner form): one ugx_line per line whose first find_in_line result is a match, or with
// lflags & UGX_LINES_INVERT per line where it is none; lflags & SCAN_LINES_NEVER: the pattern admits no candidate at all,
// no line is searched
template <int MODE, bool EMIT, bool HAS_META, int THREADS, bool LINES = false>
#ifndef UGX_SCAN_MINB
#define UGX_SCAN_MINB 8
#endif
__global__ void __launch_bounds__(THREADS, THREADS > 256 ? 2048 / THREADS : UGX_SCAN_MINB)
scan_lines_kernel(const __grid_constant__ DevPattern P, const uint8_t* __restrict__ buf, uint64_t n, uint64_t ntiles,
                  uint32_t stage_table, uint64_t* __restrict__ tile_matches, uint64_t* __restrict__ tile_newlines,
                  uint32_t* __restrict__ strip_counts, ugx_match* __restrict__ out, uint64_t out_cap,
                  uint64_t base_offset, uint64_t base_line, ugx_line* __restrict__ lout, uint32_t lflags)
{
  constexpr uint32_t TILE = THREADS * SCAN_STRIP;          // bytes per CTA iteration
  constexpr uint32_t LINE_CAP = THREADS * 4;               // line starts per tile the dense line list holds
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ uint32_t warp_sums[33];
  // ---- stage the tables: class map, predictor, bitap pairs, and the transition table when it fits ----
  uint8_t* s_cls = smem;
  uint8_t* s_pred = smem + 256;
  uint8_t* s_tap = s_pred + UGX_HASH;
  uint32_t* s_cand = reinterpret_cast<uint32_t*>(s_tap + UGX_BTAP);
  uint32_t* s_nl = s_cand + TILE / 32;
  uint16_t* s_lines = reinterpret_cast<uint16_t*>(s_nl + TILE / 32);
  uint16_t* s_next = s_lines + LINE_CAP;
  // tables -> shared memory by bulk asynchronous copies (ptx.cuh)
  __shared__ __align__(8) uint64_t s_bar;
  stage_tables_bulk(&s_bar, s_cls, P.cls, s_pred, P.pred, s_tap, P.tap, s_next, P.next,
                    stage_table ? ((P.table_bytes + 15) / 16) * 16 : 0);
  __syncthreads();
  Tables T;
  T.cls = s_cls;
  T.pred = s_pred;
  T.tap = s_tap;
  T.next = stage_table ? s_next : P.next;
  Text t{buf, n};

  for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
  {
    const uint64_t tile_base = tile * TILE;
    const uint64_t s0 = tile_base + static_cast<uint64_t>(threadIdx.x) * SCAN_STRIP;
    // ---- phase A: candidate and newline bitmaps of the tile (position-parallel prefilter)
    tile_phase_a<TILE / 16 / THREADS>(t, P, T, tile_base, reinterpret_cast<uint16_t*>(s_cand),
                                                reinterpret_cast<uint16_t*>(s_nl));
    __syncthreads();
    const CandMap cm{s_cand, tile_base, TILE};
    // ---- newline mask of my strip and the line starts in it ----
    const uint64_t nl = (static_cast<uint64_t>(s_nl[2 * threadIdx.x + 1]) << 32) | s_nl[2 * threadIdx.x];
    uint64_t starts = nl << 1;
    if (s0 < n && (s0 == 0 || __ldg(buf + s0 - 1) == '\n'))
      starts |= 1ull;
    if (s0 + SCAN_STRIP > n && s0 < n)
      starts &= (n - s0 >= 64) ? ~0ull : ((1ull << (n - s0)) - 1); // a line cannot start at or past the end
    const uint32_t my_nl = __popcll(nl);

    uint32_t strip_total = 0;
    uint64_t out_pos = 0;
    uint64_t line_no = 0;
    if (EMIT)
    {
      uint32_t cnt = s0 < n ? strip_counts[s0 / SCAN_STRIP] : 0;
      uint32_t tot;
      uint32_t ex = block_excl_scan(cnt, warp_sums, &tot);
      out_pos = tile_matches[tile] + ex;
      uint32_t nlex = block_excl_scan(my_nl, warp_sums, &tot);
      line_no = tile_newlines[tile] + nlex + 1 + base_line;
    }

    // ---- lines -> threads.  Counting without records: the tile's line starts are compacted into shared memory
    // and handed out densely (thread i takes lines i, i + 256, ...), so nearly every lane has a line to run; the
    // strip-owner assignment (a thread runs the lines that start in its 64-byte strip) is kept for record
    // passes, whose output offsets are per strip, and for tiles with more line starts than the list holds.
    bool dense = false;
    if (!EMIT && strip_counts == nullptr)
    {
      uint32_t total_lines;
      const uint32_t first_idx = block_excl_scan(static_cast<uint32_t>(__popcll(starts)), warp_sums, &total_lines);
      if (total_lines <= LINE_CAP)
      {
        dense = true;
        uint32_t idx = first_idx;
        uint64_t rest = starts;
        while (rest != 0)
        {
          const uint32_t bit = __ffsll(static_cast<long long>(rest)) - 1;
          rest &= rest - 1;
          s_lines[idx++] = static_cast<uint16_t>(threadIdx.x * SCAN_STRIP + bit);
        }
        __syncthreads();
        constexpr uint32_t NW = TILE / 32;
        for (uint32_t i = threadIdx.x; i < total_lines; i += blockDim.x)
        {
          const uint32_t off = s_lines[i];
          const uint64_t L = tile_base + off;
          // end of the line: the next newline in the tile's bitmap, else walk on in global memory
          uint64_t last;
          {
            uint32_t wi = off >> 5;
            uint32_t word = s_nl[wi] & (0xffffffffu << (off & 31));
            while (word == 0 && ++wi < NW)
              word = s_nl[wi];
            if (word != 0)
              last = tile_base + (wi << 5) + (__ffs(word) - 1);
            else
            {
              uint64_t p = tile_base + TILE;
              while (p < n && __ldg(buf + p) != '\n')
                ++p;
              last = p < n ? p : n - 1;
            }
            if (last >= n)
              last = n - 1;
          }
          Cursor m;
          set_current(t, m, L);
          for (;;)
          {
            if (find_in_line<HAS_META>(t, P, T, cm, m, last) == 0)
              break;
            ++strip_total;
            if (MODE == 0)
              break;
          }
        }
      }
    }
    if (!dense)
    {
      // ---- every line that starts in my strip ----
      uint64_t rest = starts;
      while (rest != 0)
      {
        const uint32_t bit = __ffsll(static_cast<long long>(rest)) - 1;
        rest &= rest - 1;
        const uint64_t L = s0 + bit;
        // end of the line: its '\n', or the last byte of the buffer
        uint64_t last;
        {
          const uint64_t after = nl >> bit; // newlines at or after L inside the strip
          if (after != 0)
            last = L + (__ffsll(static_cast<long long>(after)) - 1);
          else
          {
            uint64_t p = s0 + SCAN_STRIP;
            while (p < n && __ldg(buf + p) != '\n')
              ++p;
            last = p < n ? p : n - 1;
          }
        }
        uint64_t this_line = 0;
        if (EMIT)
          this_line = line_no + __popcll(nl & ((1ull << bit) - 1));
        Cursor m;
        set_current(t, m, L);
        if (LINES)
        {
          // the `ugrep -c` loop's view of the line: its first find, then on to the next line
          const uint32_t cap = (lflags & SCAN_LINES_NEVER) ? 0u : find_in_line<HAS_META>(t, P, T, cm, m, last);
          const bool inv = (lflags & UGX_LINES_INVERT) != 0;
          if ((cap != 0) != inv)
          {
            if (EMIT)
            {
              const uint64_t idx = out_pos + strip_total;
              if (idx < out_cap)
              {
                ugx_line r;
                r.line = this_line;
                r.bol = L + base_offset;
                r.eol = (__ldg(buf + last) == '\n' ? last : n) + base_offset;
                r.offset = inv ? r.bol : m.txt + base_offset;
                r.len = inv ? 0u : m.len;
                r.cap = cap;
                lout[idx] = r;
              }
            }
            ++strip_total;
          }
          continue;
        }
        for (;;)
        {
          uint32_t cap = find_in_line<HAS_META>(t, P, T, cm, m, last);
          if (cap == 0)
            break;
          if (EMIT)
          {
            uint64_t idx = out_pos + strip_total;
            if (idx < out_cap)
            {
              ugx_match r;
              r.line = this_line;
              r.offset = m.txt + base_offset;
              r.len = m.len;
              r.cap = cap;
              out[idx] = r;
            }
          }
          ++strip_total;
          if (MODE == 0)
            break;
        }
      }
    }

    if (!EMIT)
    {
      if (strip_counts != nullptr && s0 < n)
        strip_counts[s0 / SCAN_STRIP] = strip_total;
      // tile totals
      uint32_t tm = strip_total, tn = my_nl;
#pragma unroll
      for (int d = 16; d > 0; d >>= 1)
      {
        tm += __shfl_down_sync(0xffffffffu, tm, d);
        tn += __shfl_down_sync(0xffffffffu, tn, d);
      }
      __shared__ uint32_t red_m[THREADS / 32], red_n[THREADS / 32];
      if ((threadIdx.x & 31) == 0)
      {
        red_m[threadIdx.x >> 5] = tm;
        red_n[threadIdx.x >> 5] = tn;
      }
      __syncthreads();
      if (threadIdx.x == 0)
      {
        uint64_t a = 0, b = 0;
        for (uint32_t w = 0; w < blockDim.x / 32; ++w)
        {
          a += red_m[w];
          b += red_n[w];
        }
        tile_matches[tile] = a;
        tile_newlines[tile] = b;
      }
    }
    __syncthreads(); // the bitmaps are rewritten by the next tile
  }
}

// ---- launch helpers ----

inline size_t scan_smem_bytes(const DevPattern& P, bool stage, int threads)
{
  return 256 + UGX_HASH + UGX_BTAP + 2 * (threads * SCAN_STRIP / 8) + 2 * (threads * 4) + (stage ? ((P.table_bytes + 15) / 16) * 16 : 0);
}

#ifndef UGX_SCAN_BIG_THREADS
#define UGX_SCAN_BIG_THREADS 1024
#endif
template <int MODE, bool EMIT, bool HAS_META, int THREADS, bool LINES = false>
inline cudaError_t launch_one(const DevPattern& P, const ScanArgs& a, bool stage, int grid, size_t smem, cudaStream_t st,
                              ugx_line* lout = nullptr, uint32_t lflags = 0)
{
  auto kern = scan_lines_kernel<MODE, EMIT, HAS_META, THREADS, LINES>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, UGX_MAX_DYN_SMEM);
  if (e != cudaSuccess)
    return e;
  kern<<<grid, THREADS, smem, st>>>(P, a.buf, a.n, a.ntiles, stage ? 1u : 0u, a.tile_matches, a.tile_newlines,
                                         a.strip_counts, a.out, a.out_cap, a.base_offset, a.base_line, lout, lflags);
  return cudaGetLastError();
}

// persistent grid of the line-scan kernels: as many CTAs as fit per SM, times the SM count, capped by the number of tiles
inline int scan_grid(const ScanArgs& a, size_t smem, int threads, int sm_count)
{
  int per_sm = static_cast<int>((220 * 1024) / (smem + 1024));
  if (per_sm > 2048 / threads)
    per_sm = 2048 / threads;
  if (per_sm < 1)
    per_sm = 1;
  uint64_t g = static_cast<uint64_t>(sm_count) * per_sm;
  if (g > a.ntiles)
    g = a.ntiles;
  if (g == 0)
    g = 1;
  return static_cast<int>(g);
}

} // namespace ugx
