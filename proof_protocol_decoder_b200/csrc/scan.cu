// scan.cu — the exclusive prefix sums of every kernel family.
//   exclusive_scan        K arrays of u32 or u64 at a stride, in three phases: a block scan of 1024 elements per thread
//                         block, the same scan recursively over the block sums, and a pass adding the scanned sums back
//   exclusive_scan_small  one bin array of at most 4096 words in place, one launch (the counting sorts' bins)
#include <cstdint>

#include "ppd_kernels.h"
#include "scan.cuh"

namespace ppd {

static constexpr int SCAN_B = 256, SCAN_ITEMS = 4, SCAN_ELEMS = SCAN_B * SCAN_ITEMS;

// array k = blockIdx.y; block_sums[k * sums_stride + blockIdx.x] = the sum of this block's elements (when given)
template <class T>
__global__ void __launch_bounds__(SCAN_B) scan_block_kernel(const T* __restrict__ in, T* __restrict__ out, uint32_t n, size_t stride,
                                                            T* __restrict__ block_sums, size_t sums_stride) {
  __shared__ T warp_sums[SCAN_B / 32];
  const uint32_t k = blockIdx.y, lane = threadIdx.x & 31;
  in += k * stride, out += k * stride;
  uint32_t base = blockIdx.x * SCAN_ELEMS + threadIdx.x * SCAN_ITEMS;
  T v[SCAN_ITEMS], sum = 0;
#pragma unroll
  for (int q = 0; q < SCAN_ITEMS; q++) {
    v[q] = base + q < n ? in[base + q] : T(0);
    sum += v[q];
  }
  const T incl = warp_inclusive_scan(sum, lane);
  if (lane == 31) warp_sums[threadIdx.x >> 5] = incl;
  __syncthreads();
  if (threadIdx.x < 32) {
    const T ws = threadIdx.x < SCAN_B / 32 ? warp_sums[threadIdx.x] : T(0), wi = warp_inclusive_scan(ws, threadIdx.x);
    if (threadIdx.x < SCAN_B / 32) warp_sums[threadIdx.x] = wi - ws;
    if (threadIdx.x == SCAN_B / 32 - 1 && block_sums) block_sums[k * sums_stride + blockIdx.x] = wi;
  }
  __syncthreads();
  T excl = incl - sum + warp_sums[threadIdx.x >> 5];
#pragma unroll
  for (int q = 0; q < SCAN_ITEMS; q++) {
    if (base + q < n) out[base + q] = excl;
    excl += v[q];
  }
}

template <class T>
__global__ void __launch_bounds__(SCAN_B) scan_add_kernel(T* __restrict__ out, uint32_t n, size_t stride, const T* __restrict__ block_offsets,
                                                          size_t sums_stride) {
  const uint32_t k = blockIdx.y;
  out += k * stride;
  const T add = block_offsets[k * sums_stride + blockIdx.x];
  uint32_t i = blockIdx.x * SCAN_ELEMS + threadIdx.x;
#pragma unroll
  for (int q = 0; q < SCAN_ITEMS; q++) {
    uint32_t j = i + q * SCAN_B;
    if (j < n) out[j] += add;
  }
}

// exclusive scan of bins[0 .. n_bins) in place, one CTA (n_bins <= 4096)
__global__ void __launch_bounds__(1024) scan_small_kernel(uint32_t* __restrict__ bins, uint32_t n_bins) {
  __shared__ uint32_t warp_sums[32];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < n_bins; base += 1024) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < n_bins ? bins[i] : 0u;
    const uint32_t incl = warp_inclusive_scan(v, threadIdx.x & 31);
    if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
      const uint32_t ws = warp_sums[threadIdx.x];
      warp_sums[threadIdx.x] = warp_inclusive_scan(ws, threadIdx.x) - ws;
    }
    __syncthreads();
    const uint32_t excl = carry + warp_sums[threadIdx.x >> 5] + incl - v;
    if (i < n_bins) bins[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
}

size_t scan_tmp_words(size_t n, uint32_t K) {
  size_t total = 0;
  while (n > 1) {
    n = (n + SCAN_ELEMS - 1) / SCAN_ELEMS;
    total += K * ((n + 3) & ~(size_t)3);
  }
  return total + 16;
}

template <class T>
uint32_t exclusive_scan(const T* in, T* out, uint32_t n, T* tmp, cudaStream_t st, uint32_t K, size_t stride) {
  if (!n) return 0;
  uint32_t nb = (n + SCAN_ELEMS - 1) / SCAN_ELEMS, launches = 1;
  size_t ss = (nb + 3) & ~(size_t)3;
  scan_block_kernel<T><<<dim3(nb, K), SCAN_B, 0, st>>>(in, out, n, stride, nb > 1 ? tmp : nullptr, ss);
  if (nb > 1) {
    launches += exclusive_scan<T>(tmp, tmp, nb, tmp + K * ss, st, K, ss);
    scan_add_kernel<T><<<dim3(nb, K), SCAN_B, 0, st>>>(out, n, stride, tmp, ss);
    launches++;
  }
  return launches;
}
template uint32_t exclusive_scan<uint32_t>(const uint32_t*, uint32_t*, uint32_t, uint32_t*, cudaStream_t, uint32_t, size_t);
template uint32_t exclusive_scan<uint64_t>(const uint64_t*, uint64_t*, uint32_t, uint64_t*, cudaStream_t, uint32_t, size_t);

void exclusive_scan_small(uint32_t* bins, uint32_t n_bins, cudaStream_t st) { scan_small_kernel<<<1, 1024, 0, st>>>(bins, n_bins); }

}  // namespace ppd
