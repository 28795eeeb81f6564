// scan.cuh — the warp-level prefix sum under the scans of scan.cu and the block-local scans of other kernels
#pragma once
#include <cstdint>

namespace ppd {

// inclusive prefix sum of v over the 32 lanes of a converged warp; lane = this thread's lane
template <class T>
__device__ __forceinline__ T warp_inclusive_scan(T v, uint32_t lane) {
  for (int off = 1; off < 32; off <<= 1) {
    const T t = __shfl_up_sync(0xffffffffu, v, off);
    if (lane >= (uint32_t)off) v += t;
  }
  return v;
}

}  // namespace ppd
