// scan_kernels.cu — sm_100a scan kernels of the buffer-scan path.
//
// Work decomposition (DESIGN.md "line-parallel scan"): no DFA in scope has a transition
// on '\n' and the look-back set never contains '\n' (checked at pattern upload), so every
// line is an independent unit of Matcher::match(FIND) (lib/matcher.cpp:42-750).  The buffer
// is cut into 64-byte strips; a thread owns every line that STARTS in its strip and runs the
// reference's find loop on it: prefilter candidate -> look-back -> DFA -> resume.
//
// Kernels here:
//   scan_lines_kernel    generic exact line scan (all prefilter families, look-back, META, W; scan_lines.cuh)
//   tile_prefix_kernel   exclusive prefix of per-tile match / newline counts (+ totals)
// Records (ugrep -o) come from a second run of scan_lines_kernel that knows every strip's
// output offset: deterministic input order, no atomics in the ordering.
#include "scan_lines.cuh"
#include "block_scan.cuh"

namespace ugx {

// exclusive prefix over the tiles (in place) + grand totals; one block
__global__ void __launch_bounds__(1024)
tile_prefix_kernel(uint64_t* __restrict__ tile_matches, uint64_t* __restrict__ tile_newlines, uint64_t ntiles,
                   unsigned long long* __restrict__ totals)
{
  __shared__ uint64_t sm[1024], sn[1024];
  const uint64_t per = (ntiles + blockDim.x - 1) / blockDim.x;
  const uint64_t lo = threadIdx.x * per;
  const uint64_t hi = lo + per < ntiles ? lo + per : ntiles;
  uint64_t a = 0, b = 0;
  for (uint64_t i = lo; i < hi; ++i)
  {
    a += tile_matches[i];
    b += tile_newlines[i];
  }
  sm[threadIdx.x] = a;
  sn[threadIdx.x] = b;
  __syncthreads();
  if (threadIdx.x == 0)
  {
    uint64_t ra = 0, rb = 0;
    for (uint32_t i = 0; i < blockDim.x; ++i)
    {
      uint64_t x = sm[i], y = sn[i];
      sm[i] = ra;
      sn[i] = rb;
      ra += x;
      rb += y;
    }
    totals[0] = ra;
    totals[1] = rb;
  }
  __syncthreads();
  a = sm[threadIdx.x];
  b = sn[threadIdx.x];
  for (uint64_t i = lo; i < hi; ++i)
  {
    uint64_t x = tile_matches[i], y = tile_newlines[i];
    tile_matches[i] = a;
    tile_newlines[i] = b;
    a += x;
    b += y;
  }
}

// ---- launchers ----

// CTA size: a staged table of more than 40 KiB leaves room for two CTAs per SM at most — make them big.  The find
// loop is latency-bound (dependent byte loads, divergent branches): resident warps matter more than registers.
int scan_threads(const DevPattern& P)
{
  return (P.has_meta == 0 && P.table_bytes <= SCAN_MAX_SMEM_TABLE && P.table_bytes > 40 * 1024) ? UGX_SCAN_BIG_THREADS : 256;
}

uint32_t scan_tile_bytes(const DevPattern& P) { return static_cast<uint32_t>(scan_threads(P)) * SCAN_STRIP; }

cudaError_t launch_scan_lines(const DevPattern& P, const ScanArgs& a, int mode, bool emit, int sm_count, cudaStream_t st)
{
  const int threads = scan_threads(P);
  const bool stage = P.has_meta == 0 && P.table_bytes <= SCAN_MAX_SMEM_TABLE &&
                     scan_smem_bytes(P, true, threads) <= static_cast<size_t>(UGX_MAX_DYN_SMEM);
  const size_t smem = scan_smem_bytes(P, stage, threads);
  const int grid = scan_grid(a, smem, threads, sm_count);
  const bool meta = P.has_meta != 0;
#define UGX_SCAN_GO(MODE, EMIT)                                                                                 \
  do                                                                                                            \
  {                                                                                                             \
    if (meta)                                                                                                   \
      return launch_one<MODE, EMIT, true, 256>(P, a, stage, grid, smem, st);                                    \
    if (threads != 256)                                                                                         \
      return launch_one<MODE, EMIT, false, UGX_SCAN_BIG_THREADS>(P, a, stage, grid, smem, st);                                   \
    return launch_one<MODE, EMIT, false, 256>(P, a, stage, grid, smem, st);                                     \
  } while (0)
  if (mode == 0)
    UGX_SCAN_GO(0, false);
  if (!emit)
    UGX_SCAN_GO(1, false);
  UGX_SCAN_GO(1, true);
#undef UGX_SCAN_GO
}

cudaError_t launch_tile_prefix(uint64_t* tile_matches, uint64_t* tile_newlines, uint64_t ntiles,
                               unsigned long long* totals, cudaStream_t st)
{
  tile_prefix_kernel<<<1, 1024, 0, st>>>(tile_matches, tile_newlines, ntiles, totals);
  return cudaGetLastError();
}

} // namespace ugx
