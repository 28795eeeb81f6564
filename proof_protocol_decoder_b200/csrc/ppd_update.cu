// ppd_update.cu — an update of a resident trie (ppd_trie_update[_dev], csrc/gpu_trie.cu): merge a sorted batch of writes
// and deletes into the trie's sorted leaves, then re-hash only what the batch changed.
//
// A trie's shape depends only on its keys.  After the builder's structure passes (ppd_build.cu) have run on the merged
// leaves, a node whose subtree holds no key of the batch is the node it was before, at a new id:
//   leaf i      clean when it is an old leaf (src[i]) whose parent depth max(L[i], L[i + 1]) did not change: its
//               encoding is its key from that depth on, and its value;
//   branch b    not marked by a walk of some batch key (subset_mark_kernel marks exactly the branches whose prefix a
//               batch key shares): its leaves are those of the old branch whose leader sits where its own leader's leaf
//               sat.  Clean when its extension also starts where it did.
// Clean nodes copy ref / ref_len (and a branch inner_ref / inner_ref_len) from the old trie; the rest are hashed.
#include <cstdint>

#include "build_leaf.cuh"
#include "ppd_kernels.h"

namespace ppd {

static constexpr uint32_t FULL = 0xffffffffu;

// key at p as big-endian words (p need not be 16-byte aligned: keys the caller hands in unhashed)
__device__ __forceinline__ void load_key_be(const uint8_t* p, uint32_t w[8]) {
  if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(p)), b = __ldg(reinterpret_cast<const uint4*>(p) + 1);
    const uint32_t x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int k = 0; k < 8; k++) w[k] = __byte_perm(x[k], 0, 0x0123);
  } else {
#pragma unroll
    for (int k = 0; k < 8; k++)
      w[k] = ((uint32_t)__ldg(p + 4 * k) << 24) | ((uint32_t)__ldg(p + 4 * k + 1) << 16) | ((uint32_t)__ldg(p + 4 * k + 2) << 8) | __ldg(p + 4 * k + 3);
  }
}

// sign of (key at p) - q
__device__ __forceinline__ int cmp_key(const uint8_t* p, const uint32_t q[8]) {
  uint32_t w[8];
  load_key_be(p, w);
#pragma unroll
  for (int k = 0; k < 8; k++)
    if (w[k] != q[k]) return w[k] < q[k] ? -1 : 1;
  return 0;
}

// ------------------------------------------------------------------ merge -----------------------------------------------

// sorted position j of the batch, when it is the last occurrence of its key: its lower bound p in the old leaves.
// Drops old leaf p when the key is there (overwritten or deleted); a write is inserted before old leaf p.
__global__ void merge_locate_kernel(MergeView M) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j > M.k) return;
  if (j == M.k) {
    M.written[j] = 0;
    return;
  }
  uint32_t w = 0;
  if (M.keep[j]) {
    const uint32_t u = M.idx[j];
    uint32_t q[8];
    load_key_be(M.ukeys32 + 32ull * u, q);
    uint32_t lo = 0, hi = M.n_old;
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (cmp_key(M.okeys + 32ull * mid, q) < 0)
        lo = mid + 1;
      else
        hi = mid;
    }
    if (lo < M.n_old && cmp_key(M.okeys + 32ull * lo, q) == 0) M.drop[lo] = 1;
    w = !(M.del && M.del[u]);
    if (w) atomicAdd(M.ins + lo, 1u);
    M.upos[j] = lo;
  }
  M.written[j] = w;
}

// every leaf of the merged set at its position: src[i] = its old position, or MERGE_SRC_UPD | its sorted batch position;
// len[i] = its value's length (len[n_new] = 0: the scan's last element)
__global__ void merge_place_kernel(MergeView M) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t == 0) M.len[M.n_new] = 0;
  if (t < M.n_old) {
    const uint32_t p = (uint32_t)t;
    if (M.drop[p]) return;
    const uint32_t at = p - M.dpos[p] + M.ipos[p + 1];  // kept old leaves before it, and every write whose key is smaller
    M.src[at] = p;
    M.len[at] = M.ooff[p + 1] - M.ooff[p];
  } else if (t < (uint64_t)M.n_old + M.k) {
    const uint32_t j = (uint32_t)(t - M.n_old);
    if (M.wpos[j + 1] == M.wpos[j]) return;
    const uint32_t p = M.upos[j], u = M.idx[j];
    const uint32_t at = p - M.dpos[p] + M.wpos[j];
    M.src[at] = MERGE_SRC_UPD | j;
    M.len[at] = M.uoff[u + 1] - M.uoff[u];
  }
}

// n bytes from src to dst (any alignment) by the 32 lanes of a warp: 32-bit stores once dst is aligned, each assembled
// from the two aligned source words it straddles
__device__ __forceinline__ void warp_copy(uint8_t* dst, const uint8_t* src, uint64_t n, uint32_t lane) {
  const uint64_t align = (4 - (reinterpret_cast<uintptr_t>(dst) & 3)) & 3, head = align < n ? align : n;
  if (lane < head) dst[lane] = __ldg(src + lane);
  dst += head, src += head, n -= head;
  const uintptr_t a = reinterpret_cast<uintptr_t>(src);
  const uint32_t* q = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3) * 8;
  uint32_t* d = reinterpret_cast<uint32_t*>(dst);
  const uint64_t words = n >> 2;
  for (uint64_t k = lane; k < words; k += 32) {
    const uint32_t lo = __ldg(q + k), hi = sh ? __ldg(q + k + 1) : 0u;
    d[k] = __funnelshift_r(lo, hi, sh);
  }
  const uint32_t r = (uint32_t)(n & 3);
  if (lane < r) dst[4 * words + lane] = __ldg(src + 4 * words + lane);
}

// n bytes by one thread (as gather_kernel of ppd_leaves.cu)
__device__ __forceinline__ void thread_copy(uint8_t* dst, const uint8_t* src, uint64_t n) {
  for (; n && (reinterpret_cast<uintptr_t>(dst) & 3); n--) *dst++ = __ldg(src++);
  const uintptr_t a = reinterpret_cast<uintptr_t>(src);
  const uint32_t* q = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3) * 8;
  uint32_t* d = reinterpret_cast<uint32_t*>(dst);
  const uint64_t words = n >> 2;
  for (uint64_t k = 0; k < words; k++) d[k] = __funnelshift_r(__ldg(q + k), sh ? __ldg(q + k + 1) : 0u, sh);
  dst += 4 * words, src += 4 * words;
  for (uint32_t r = (uint32_t)(n & 3); r; r--) *dst++ = __ldg(src++);
}

// keys and values of the merged leaves.  A warp takes 32 consecutive leaves: when their bytes come from one place in
// the same order (a run of kept old leaves: every lane's source sits at the same distance from its destination) the
// warp copies the whole range together; otherwise (a run broken by a write or a dropped leaf) each lane copies its own.
__global__ void __launch_bounds__(256) merge_copy_kernel(MergeView M) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
  if (i - lane >= M.n_new) return;  // (warp-uniform)
  const bool live = i < M.n_new;
  const uint8_t* vs = nullptr;
  uint64_t vd = 0, vlen = 0;
  if (live) {
    const uint32_t s = M.src[i];
    const uint8_t* ks;
    uint64_t b;
    if (s & MERGE_SRC_UPD) {
      const uint32_t u = M.idx[s & ~MERGE_SRC_UPD];
      ks = M.ukeys32 + 32ull * u;
      b = M.uoff[u], vlen = M.uoff[u + 1] - b, vs = M.uvals + b;
    } else {
      ks = M.okeys + 32ull * s;
      b = M.ooff[s], vlen = M.ooff[s + 1] - b, vs = M.ovals + b;
    }
    uint4* ko = reinterpret_cast<uint4*>(M.nkeys + 32ull * i);
    if ((reinterpret_cast<uintptr_t>(ks) & 15) == 0)
      ko[0] = __ldg(reinterpret_cast<const uint4*>(ks)), ko[1] = __ldg(reinterpret_cast<const uint4*>(ks) + 1);
    else
      thread_copy(M.nkeys + 32ull * i, ks, 32);
    vd = M.noff[i];
  }
  const long long delta = live ? (long long)(reinterpret_cast<uintptr_t>(vs) - reinterpret_cast<uintptr_t>(M.nvals + vd)) : 0;
  const long long delta0 = __shfl_sync(FULL, delta, 0);
  if (__all_sync(FULL, !live || delta == delta0)) {
    const uint32_t last = 31 - __clz(__ballot_sync(FULL, live));
    const uint64_t lo = __shfl_sync(FULL, vd, 0), hi = __shfl_sync(FULL, vd + vlen, last);
    warp_copy(M.nvals + lo, M.nvals + lo + delta0, hi - lo, lane);
  } else if (live) {
    thread_copy(M.nvals + vd, vs, vlen);
  }
}

// ------------------------------------------------------------------ incremental hashing ---------------------------------

// Places leaf i in the new trie (as the leaf hasher does), then copies its ref when it is clean, or lists it for the
// hasher (hash_sorted_leaves_kernel with a LeafList).
__global__ void __launch_bounds__(256) update_leaves_kernel(BuildView V, OldTrie O, const uint32_t* __restrict__ src, uint32_t* __restrict__ list,
                                                            uint32_t* __restrict__ count) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
  bool dirty = false;
  if (i < V.n) {
    const Pyramid& P = V.P;
    int dl = P.L[i], dr = P.L[i + 1];
    int dp = max(dl, dr);
    const uint8_t* key = V.keys + 32ull * i;
    const bool is_root = dp < V.base_depth;
    place_leaf(V, i, dl, dr, dp, key, is_root);
    const uint32_t s = src[i];
    dirty = (s & MERGE_SRC_UPD) || max((int)O.L[s], (int)O.L[s + 1]) != dp;
    if (!dirty) {
      const uint4* r = reinterpret_cast<const uint4*>(O.ref + 32ull * s);
      const uint4 x = r[0], y = r[1];
      uint4* o = reinterpret_cast<uint4*>(V.ref + 32ull * i);
      o[0] = x, o[1] = y;
      V.ref_len[i] = O.ref_len[s];
      if (is_root) {
        uint4* ro = reinterpret_cast<uint4*>(V.root_out);
        ro[0] = x, ro[1] = y;
      }
    }
  }
  const uint32_t ballot = __ballot_sync(FULL, dirty);
  uint32_t base = 0;
  if (lane == 0 && ballot) base = atomicAdd(count, (uint32_t)__popc(ballot));
  base = __shfl_sync(FULL, base, 0);
  if (dirty) list[base + __popc(ballot & ((1u << lane) - 1))] = i;
}

// Branch b (leader q): clean when no batch key marked it and the old branch with the same leaves has its extension
// start; a clean branch copies its refs and gets the CLEAN tag in nchild[b] (the counting sort's key: UpdateBranchKey).
__global__ void __launch_bounds__(256) update_branches_kernel(BuildView V, OldTrie O, const uint32_t* __restrict__ src, const uint32_t* __restrict__ bits,
                                                              uint32_t* __restrict__ nchild) {
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q == 0 || q >= V.n) return;
  if (V.leader[q] != q) return;
  const uint32_t b = V.bidx[q];
  const uint64_t mark = (uint64_t)V.n + b;
  if ((bits[mark >> 5] >> (mark & 31)) & 1u) return;
  // the old leader sits between the old leaves of leaves q - 1 and q, when both are old leaves next to each other
  const uint32_t s = src[q], s0 = src[q - 1];
  if ((s & MERGE_SRC_UPD) || (s0 & MERGE_SRC_UPD) || s0 + 1 != s || O.leader[s] != s) return;
  const uint32_t ob = O.bidx[s];
  if (O.depth[ob] != V.depth[b] || O.ext_start[ob] != V.ext_start[b]) return;
  const uint4* r = reinterpret_cast<const uint4*>(O.ref + 32ull * (O.n + ob));
  const uint4 x = r[0], y = r[1];
  uint4* o = reinterpret_cast<uint4*>(V.ref + 32ull * (V.n + b));
  o[0] = x, o[1] = y;
  V.ref_len[V.n + b] = O.ref_len[O.n + ob];
  const uint4* ir = reinterpret_cast<const uint4*>(O.inner_ref + 32ull * ob);
  uint4* io = reinterpret_cast<uint4*>(V.inner_ref + 32ull * b);
  io[0] = ir[0], io[1] = ir[1];
  V.inner_ref_len[b] = O.inner_ref_len[ob];
  if (*V.root_id == V.n + b) {
    uint4* ro = reinterpret_cast<uint4*>(V.root_out);
    ro[0] = x, ro[1] = y;
  }
  nchild[b] |= BRANCH_CLEAN;
}

// ------------------------------------------------------------------ launchers -------------------------------------------
static inline uint32_t grid(uint64_t n, uint32_t b) { return (uint32_t)((n + b - 1) / b); }

void launch_merge_locate(const MergeView& M, cudaStream_t st) { merge_locate_kernel<<<grid((uint64_t)M.k + 1, 256), 256, 0, st>>>(M); }
void launch_merge_place(const MergeView& M, cudaStream_t st) {
  merge_place_kernel<<<grid(std::max<uint64_t>((uint64_t)M.n_old + M.k, 1), 256), 256, 0, st>>>(M);
}
void launch_merge_copy(const MergeView& M, cudaStream_t st) {
  if (M.n_new) merge_copy_kernel<<<grid(M.n_new, 256), 256, 0, st>>>(M);
}
void launch_update_leaves(const BuildView& V, const OldTrie& O, const uint32_t* src, uint32_t* list, uint32_t* count, cudaStream_t st) {
  if (V.n) update_leaves_kernel<<<grid(V.n, 256), 256, 0, st>>>(V, O, src, list, count);
}
void launch_update_branches(const BuildView& V, const OldTrie& O, const uint32_t* src, const uint32_t* bits, uint32_t* nchild, cudaStream_t st) {
  if (V.n >= 2) update_branches_kernel<<<grid(V.n, 256), 256, 0, st>>>(V, O, src, bits, nchild);
}

}  // namespace ppd
