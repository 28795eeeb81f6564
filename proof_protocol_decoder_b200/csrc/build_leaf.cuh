// build_leaf.cuh — where a leaf of the sorted-leaf builder (ppd_build.cu) sits: shared by the leaf hasher and by an
// update's leaf pass (ppd_update.cu), which both register the leaf with its parent.
#pragma once
#include <cstdint>

#include "ppd_kernels.h"

namespace ppd {

// Leaf i's parent is the branch owning position i or i + 1, whichever has the larger L (dl = L[i], dr = L[i + 1], dp =
// max of them: the parent's depth); when dp is above base_depth the leaf is the root.  Registers the leaf in its
// parent's child table, or as the root.  key: leaf i's key.
__device__ __forceinline__ void place_leaf(const BuildView& V, uint32_t i, int dl, int dr, int dp, const uint8_t* key, bool is_root) {
  if (is_root) {
    *V.root_id = i;
  } else {
    uint32_t pl = (dl >= dr) ? i : i + 1;
    uint32_t pb = V.bidx[V.leader[pl]];
    uint32_t kb = __ldg(key + (dp >> 1));
    uint32_t nib = (dp & 1) ? (kb & 15u) : (kb >> 4);
    V.child[16ull * pb + nib] = i;
  }
}

}  // namespace ppd
