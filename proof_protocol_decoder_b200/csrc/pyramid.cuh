// pyramid.cuh — nearest-smaller-value queries over an int8 array (`Pyramid`) through a 3-level min-pyramid
// (64 / 4 096 / 262 144 positions per cell).  Used by the sorted-leaf trie builder (ppd_build.cu: branch runs
// of the LCP array); the witness parser has its own int16 form with an extra 8-wide level (ppd_parse.cu,
// scan_right8).
#pragma once
#include <cstdint>

#include "ppd_kernels.h"

namespace ppd {

// largest p < q with L[p] < thr (thr >= 0; L[0] = -1 guarantees termination)
static __device__ __forceinline__ uint32_t scan_left(const Pyramid& P, uint32_t q, int thr) {
  uint32_t p = q - 1;
  for (;;) {
    if ((p & 63u) == 63u) {
      if ((p & 4095u) == 4095u) {
        if ((p & 262143u) == 262143u && P.m3[p >> 18] >= thr) {
          p -= 262144u;
          continue;
        }
        if (P.m2[p >> 12] >= thr) {
          p -= 4096u;
          continue;
        }
      }
      if (P.m1[p >> 6] >= thr) {
        p -= 64u;
        continue;
      }
    }
    if (P.L[p] < thr) return p;
    p--;
  }
}
// smallest r > q with L[r] < thr (L[N] = -1 guarantees termination)
static __device__ __forceinline__ uint32_t scan_right(const Pyramid& P, uint32_t q, int thr) {
  uint32_t p = q + 1;
  for (;;) {
    if ((p & 63u) == 0u) {
      if ((p & 4095u) == 0u) {
        if ((p & 262143u) == 0u && P.m3[p >> 18] >= thr) {
          p += 262144u;
          continue;
        }
        if (P.m2[p >> 12] >= thr) {
          p += 4096u;
          continue;
        }
      }
      if (P.m1[p >> 6] >= thr) {
        p += 64u;
        continue;
      }
    }
    if (P.L[p] < thr) return p;
    p++;
  }
}

}  // namespace ppd
