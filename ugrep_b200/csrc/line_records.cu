// line_records.cu — the line-record instantiations of scan_lines_kernel (ugx_find_lines, general route): a count
// pass into the strip counts and an emit pass that writes one ugx_line per line whose first find_in_line result is a
// match (or, inverted, is none).
#include "scan_lines.cuh"

namespace ugx {

cudaError_t launch_scan_line_records(const DevPattern& P, const ScanArgs& a, ugx_line* out, uint32_t lflags, bool emit,
                                     int sm_count, cudaStream_t st)
{
  const int threads = scan_threads(P);
  const bool stage = P.has_meta == 0 && P.table_bytes <= SCAN_MAX_SMEM_TABLE &&
                     scan_smem_bytes(P, true, threads) <= static_cast<size_t>(UGX_MAX_DYN_SMEM);
  const size_t smem = scan_smem_bytes(P, stage, threads);
  const int grid = scan_grid(a, smem, threads, sm_count);
#define UGX_LINES_GO(EMIT)                                                                                               \
  do                                                                                                                     \
  {                                                                                                                      \
    if (P.has_meta != 0)                                                                                                 \
      return launch_one<0, EMIT, true, 256, true>(P, a, stage, grid, smem, st, out, lflags);                            \
    if (threads != 256)                                                                                                  \
      return launch_one<0, EMIT, false, UGX_SCAN_BIG_THREADS, true>(P, a, stage, grid, smem, st, out, lflags);          \
    return launch_one<0, EMIT, false, 256, true>(P, a, stage, grid, smem, st, out, lflags);                             \
  } while (0)
  if (emit)
    UGX_LINES_GO(true);
  UGX_LINES_GO(false);
#undef UGX_LINES_GO
}

} // namespace ugx
