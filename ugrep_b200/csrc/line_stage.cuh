// line_stage.cuh — building blocks of the stages over line records (context_lines.cu, bool_lines.cu)
#pragma once

#include <cstdint>

namespace ugx {

// bit k = byte k of the 16 bytes at b + c is '\n' (bytes at or past end read as none)
__device__ __forceinline__ uint32_t newlines16(const uint8_t* b, uint64_t end, uint64_t c)
{
  uint32_t w[4];
  if (c + 16 <= end)
  {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(b + c));
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
      for (int j = 0; j < 4; ++j)
        if (c + 4 * k + j < end)
          w[k] |= static_cast<uint32_t>(__ldg(b + c + 4 * k + j)) << (8 * j);
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

// the last f in [lo, hi) with a[f] <= x, given a[lo] <= x and a[hi] > x (a bisection; a may repeat values)
__device__ __forceinline__ uint64_t last_le(const uint64_t* a, uint64_t lo, uint64_t hi, uint64_t x)
{
  while (hi - lo > 1)
  {
    const uint64_t mid = lo + (hi - lo) / 2;
    if (__ldg(a + mid) <= x)
      lo = mid;
    else
      hi = mid;
  }
  return lo;
}

// the grid of a grid-stride kernel: `work` items at `per` a block, at least one block and at most per_sm a multiprocessor
inline unsigned capped_grid(uint64_t work, uint64_t per, int sm_count, int per_sm)
{
  uint64_t g = (work + per - 1) / per;
  const uint64_t gmax = static_cast<uint64_t>(sm_count) * per_sm;
  if (g > gmax)
    g = gmax;
  return static_cast<unsigned>(g == 0 ? 1 : g);
}

} // namespace ugx
