// block_scan.cuh — warp / block exclusive prefix sums and block sums, over uint32_t or uint64_t.
#pragma once

#include <cstdint>

namespace ugx {

template <typename T>
__device__ __forceinline__ T warp_excl_scan(T v, uint32_t lane)
{
  T x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1)
  {
    T y = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= static_cast<uint32_t>(d))
      x += y;
  }
  return x - v;
}

// exclusive scan over the block; total returned through *total (all threads).  warp_sums[33].
template <typename T>
__device__ __forceinline__ T block_excl_scan(T v, T* warp_sums, T* total)
{
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  T ex = warp_excl_scan(v, lane);
  if (lane == 31)
    warp_sums[wid] = ex + v;
  __syncthreads();
  if (wid == 0)
  {
    T s = lane < nw ? warp_sums[lane] : 0;
    T e = warp_excl_scan(s, lane);
    if (lane < nw)
      warp_sums[lane] = e;
    if (lane == 31)
      warp_sums[32] = e + s;
  }
  __syncthreads();
  T r = ex + warp_sums[wid];
  *total = warp_sums[32];
  __syncthreads();
  return r;
}

// the sum of v over a block of THREADS threads (all threads).  sums[THREADS / 32]; a second call on the same sums
// needs a barrier before it.
template <int THREADS, typename T>
__device__ __forceinline__ T block_sum(T v, T* sums)
{
#pragma unroll
  for (int d = 16; d > 0; d >>= 1)
    v += __shfl_down_sync(0xffffffffu, v, d);
  if ((threadIdx.x & 31) == 0)
    sums[threadIdx.x >> 5] = v;
  __syncthreads();
  T all = 0;
#pragma unroll
  for (int w = 0; w < THREADS / 32; ++w)
    all += sums[w];
  return all;
}

} // namespace ugx
