// ppd_build.cu — trie construction ON THE GPU from leaves sorted by key, and the root computation
// over the resulting structure-of-arrays arena (config 5: full state-trie rehash; also the shape
// of every large storage trie).
//
// Replaces: building a HashedPartialTrie by repeated `insert` (eth_trie_utils trie_ops.rs; call
// sites compact_to_partial_trie.rs:105,125) followed by the recursive `hash()` (SURVEY.md 3.3).
//
// With the keys sorted, the Patricia trie is determined by the array L of longest common nibble
// prefixes of adjacent keys (L[i] = lcp(key[i-1], key[i]); L[0] = L[N] = -1):
//   * a branch node at depth d  <=>  a maximal run of positions q with L[q] >= d that contains at
//     least one L[q] == d; its "leader" is the leftmost position of the run with L == d;
//   * the parent of a leaf i is the branch owning position i or i+1, whichever has the larger L;
//   * the parent of a branch spanning items [l, r] is the branch owning position l or r+1,
//     whichever has the larger L; if that depth Dp < d-1 the d-Dp-1 nibbles in between form an
//     extension node, which is encoded and hashed by the same thread right after its branch.
// "Nearest position to the left/right with a smaller L" queries run on a 3-level min-pyramid
// (64 / 4096 / 262144 positions per cell), so every thread does O(64 * levels) byte reads at worst.
//
// Arena (structure of arrays, all in HBM):
//   leaves   id i in [0, N):        keys32[i], vals[val_off[i]..val_off[i+1])
//   branches id N + b, b in [0, B): depth[b], child[b][16] (ids or NODE_EMPTY), ext_start[b],
//                                   rep[b] (an item below it: its key spells the extension nibbles)
//   ref[id][32] + ref_len[id]: what the parent embeds.
// Branches are counting-sorted by depth; one launch per non-empty depth, deepest first.
#include <cstdint>

#include "arena.h"
#include "encode.cuh"
#include "keccak.cuh"
#include "build_leaf.cuh"
#include "ppd_kernels.h"
#include "pyramid.cuh"

namespace ppd {

using namespace enc;
static constexpr uint32_t FULL = 0xffffffffu;

// ------------------------------------------------------------------ structure kernels ---------

__device__ __forceinline__ int lcp_nibbles(const uint4* a, const uint4* bq, int* cmp) {
  // 32-byte big-endian keys; returns common nibble prefix and sign of (a - b) through *cmp
  const uint32_t* x = reinterpret_cast<const uint32_t*>(a);
  const uint32_t* y = reinterpret_cast<const uint32_t*>(bq);
  for (int w = 0; w < 8; w++) {
    uint32_t xv = __byte_perm(x[w], 0, 0x0123), yv = __byte_perm(y[w], 0, 0x0123);  // to big-endian order
    uint32_t diff = xv ^ yv;
    if (diff) {
      *cmp = xv < yv ? -1 : 1;
      return 8 * w + (__clz(diff) >> 2);
    }
  }
  *cmp = 0;
  return 64;
}

// L[0] = L[N] = -1;  L[i] = lcp(key[i-1], key[i]).  flags[0] |= BUILD_F_UNSORTED if not strictly ascending.
// (for a SUB-trie whose keys share their first base_depth nibbles the two ends get base_depth - 1, which is what
// they are inside the whole trie: every node then sits where it sits there.  A pair sharing fewer nibbles raises
// BUILD_F_PREFIX and stores base_depth, so that the ends stay below every interior L and the scans stay in range
// until the host rejects the input.)
__global__ void lcp_kernel(const uint8_t* __restrict__ keys, uint32_t n, int8_t* __restrict__ L, uint32_t* __restrict__ flags, int boundary) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == 0 || i == n) {
    L[i] = (int8_t)boundary;
    return;
  }
  uint4 ka[2], kb[2];
  const uint4* pa = reinterpret_cast<const uint4*>(keys + 32ull * (i - 1));
  const uint4* pb = reinterpret_cast<const uint4*>(keys + 32ull * i);
  ka[0] = __ldg(pa), ka[1] = __ldg(pa + 1), kb[0] = __ldg(pb), kb[1] = __ldg(pb + 1);
  int cmp;
  int l = lcp_nibbles(ka, kb, &cmp);
  if (cmp >= 0) atomicOr(flags, BUILD_F_UNSORTED);
  if (boundary >= 0 && l <= boundary) {
    atomicOr(flags, BUILD_F_PREFIX);
    l = boundary + 1;
  }
  L[i] = (int8_t)(l > 63 ? 63 : l);
}

// out[j] = min(in[64 j .. 64 j + 63]) over the valid entries
__global__ void min64_kernel(const int8_t* __restrict__ in, uint32_t n_in, int8_t* __restrict__ out, uint32_t n_out) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_out) return;
  int m = 127;
  uint64_t base = 64ull * j;
  for (uint32_t k = 0; k < 64 && base + k < n_in; k++) m = min(m, (int)in[base + k]);
  out[j] = (int8_t)m;
}

// link[q] = nearest position to the left in the same branch run with the same depth, else q
__global__ void link_kernel(Pyramid P, uint32_t n, uint32_t* __restrict__ link) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q == 0 || q >= n) {
    if (q == 0 || q == n) link[q] = q;
    return;
  }
  int d = P.L[q];
  uint32_t p = scan_left(P, q, d + 1);  // nearest with L <= d
  link[q] = (P.L[p] == d) ? p : q;
}
__global__ void jump_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t n_plus_1) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n_plus_1) return;
  out[q] = in[in[q]];
}
__global__ void leader_flag_kernel(const uint32_t* __restrict__ leader, uint32_t n, uint32_t* __restrict__ flag) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q > n) return;
  flag[q] = (q >= 1 && q < n && leader[q] == q) ? 1u : 0u;
}

// per leader: depth, extension, parent link
__global__ void branch_info_kernel(BuildView V) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q == 0 || q >= V.n) return;
  if (V.leader[q] != q) return;
  const Pyramid& P = V.P;
  uint32_t bi = V.bidx[q];
  int d = P.L[q];
  uint32_t l = scan_left(P, q, d);    // L[l] < d : item l is the first item of the branch
  uint32_t r1 = scan_right(P, q, d);  // L[r1] < d : item r1 - 1 is the last
  int dl = P.L[l], dr = P.L[r1];
  int dp = max(dl, dr);
  V.depth[bi] = (uint8_t)d;
  V.rep[bi] = l;
  V.ext_start[bi] = (uint8_t)(dp + 1);
  if (dp < V.base_depth) {
    *V.root_id = V.n + bi;
  } else {
    uint32_t pl = (dl >= dr) ? l : r1;
    uint32_t pb = V.bidx[V.leader[pl]];
    uint32_t b = __ldg(V.keys + 32ull * l + (dp >> 1));
    uint32_t nib = (dp & 1) ? (b & 15u) : (b >> 4);
    V.child[16ull * pb + nib] = V.n + bi;
  }
}

// nchild[b] = number of children of branch b, minus one: every position of the branch's run whose L
// equals the branch depth separates two children
__global__ void child_count_kernel(const uint32_t* __restrict__ leader, const uint32_t* __restrict__ bidx, uint32_t n, uint32_t* __restrict__ nchild) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q == 0 || q >= n) return;
  atomicAdd(nchild + bidx[leader[q]], 1u);
}

// ------------------------------------------------------------------ hashing kernels -----------
// Both kernels loop warp-uniformly: lanes fill their stage (cheap, may diverge), then the whole warp
// runs the single keccak_f1600 site converged; the loop ends when no lane has a block left.

// the leaves a launch of hash_sorted_leaves_kernel hashes: all of them, or a LeafList
__device__ __forceinline__ uint32_t leaves_of(const BuildView& V) { return V.n; }
__device__ __forceinline__ uint32_t leaves_of(const BuildView&, LeafList l) { return l.count; }
__device__ __forceinline__ uint32_t leaf_at(uint32_t slot) { return slot; }
__device__ __forceinline__ uint32_t leaf_at(uint32_t slot, LeafList l) { return slot < l.count ? l.list[slot] : 0u; }
// a leaf of the whole set is placed by the hasher; a listed leaf was placed by the update's leaf pass
__device__ __forceinline__ void place_unlisted(const BuildView& V, uint32_t i, int dl, int dr, int dp, const uint8_t* key, bool is_root) {
  place_leaf(V, i, dl, dr, dp, key, is_root);
}
__device__ __forceinline__ void place_unlisted(const BuildView&, uint32_t, int, int, int, const uint8_t*, bool, LeafList) {}

// Every leaf, each placed in its parent here; or, given a LeafList (the kernel's one extra parameter), only the leaves
// list[0 .. count), which an update's leaf pass has already placed (ppd_update.cu).  A parameter pack rather than a
// flag, so that the root entries' instantiation keeps the single BuildView parameter.
template <int B, class... Listed>
__global__ void __launch_bounds__(B, 4) hash_sorted_leaves_kernel(BuildView V, Listed... listed) {
  __shared__ uint32_t smem[PPD_STAGE_WORDS * B];
  const uint32_t i = leaf_at(blockIdx.x * B + threadIdx.x, listed...);
  uint32_t hashed = 0, perms = 0, enc_bytes = 0;
  bool busy = blockIdx.x * B + threadIdx.x < leaves_of(V, listed...), is_root = false;
  const uint8_t* key = nullptr;
  const uint8_t* val = nullptr;
  uint32_t nib_start = 0, nib_len = 0, vlen = 0, vhdr = 0, payload = 0, total = 0, nunit = 0, unit = 0;
  if (busy) {
    const Pyramid& P = V.P;
    int dl = P.L[i], dr = P.L[i + 1];
    int dp = max(dl, dr);
    key = V.keys + 32ull * i;
    is_root = dp < V.base_depth;
    place_unlisted(V, i, dl, dr, dp, key, is_root, listed...);
    nib_start = (uint32_t)(dp + 1), nib_len = 64 - nib_start;
    const uint64_t vo = V.val_off[i];
    val = V.vals + vo;
    vlen = (uint32_t)(V.val_off[i + 1] - vo);
    vhdr = (vlen == 1 && __ldg(val) < 0x80) ? 0 : len_prefix_size(vlen);
    payload = hex_prefix_str_size(nib_len) + vhdr + vlen;
    total = len_prefix_size(payload) + payload;
    nunit = 1 + ((vlen + 127) >> 7);
    if (is_root && V.base_depth > 0 && total < 32) atomicOr(V.flags, BUILD_F_SHORT_TOP);
  }
  const bool inline_ref = !is_root && total < 32;
  Stage<B> s;
  s.init(smem);
  uint64_t a[25];
#pragma unroll
  for (int k = 0; k < 25; k++) a[k] = 0;
  for (;;) {
    bool permute = false, last = false;
    if (busy) {
      while (s.bytes() < 136 && unit < nunit) {
        if (unit == 0) {
          emit_len_prefix(s, payload, 0xc0, 0xf7);
          emit_hex_prefix_str(s, key, nib_start, nib_len, 1);
          if (vhdr) emit_len_prefix(s, vlen, 0x80, 0xb7);
        } else {
          uint32_t off = (unit - 1) << 7;
          emit_bytes(s, val + off, min(128u, vlen - off));
        }
        unit++;
      }
      if (inline_ref) {
        uint4 x, y;
        inline_ref_words(s, total, x, y);
        uint4* o = reinterpret_cast<uint4*>(V.ref + 32ull * i);
        o[0] = x, o[1] = y;
        V.ref_len[i] = (uint8_t)total;
        busy = false;
      } else {
        last = s.bytes() < 136;
        if (last) s.pad();
        absorb_stage<B>(a, s);
        permute = true;
      }
    }
    if (!__any_sync(FULL, permute)) break;
    keccak_f1600(a);
    if (permute) {
      perms++;
      if (last) {
        uint4 x, y;
        digest_words(a, x, y);
        uint4* o = reinterpret_cast<uint4*>(V.ref + 32ull * i);
        o[0] = x, o[1] = y;
        V.ref_len[i] = 32;
        hashed = 1;
        enc_bytes = total;
        if (is_root) {
          uint4* ro = reinterpret_cast<uint4*>(V.root_out);
          ro[0] = x, ro[1] = y;
        }
        busy = false;
      } else {
        s.consume_block();
      }
    }
  }
  add_counters(V.counters, hashed, perms, enc_bytes);
}

// One level of branches (all at the same depth), each followed by its extension node if it has one.
// Units of the branch message: 0 = list header, 1..4 = four child slots each (4 also carries the
// empty value).  The extension message (header, hex-prefix nibbles, the branch's ref) is one unit.
// INNER: V.inner_ref is set (a compile-time switch: the root entries run the kernel without the stores)
template <int B, bool INNER>
__global__ void __launch_bounds__(B, 4) hash_branch_level_kernel(BuildView V, const uint32_t* __restrict__ order, uint32_t begin, uint32_t end) {
  __shared__ uint32_t smem[PPD_STAGE_WORDS * B];
  const uint32_t slot = begin + blockIdx.x * B + threadIdx.x;
  uint32_t hashed = 0, perms = 0, enc_bytes = 0;
  bool busy = slot < end, is_root = false;
  uint32_t bi = 0, id = 0, es = 0, ext_len = 0, payload = 1, total = 0, unit = 0, phase = 0;
  uint32_t rem = 0, hmask = 0, next_slot = 0, nunit = 0;  // slots still to emit; slots referenced by hash
  if (busy) {
    bi = __ldg(order + slot);
    id = V.n + bi;
    const uint32_t d = V.depth[bi];
    es = V.ext_start[bi];
    ext_len = d - es;
    is_root = (*V.root_id == id);
    uint32_t kid[16];
    const uint4* ct = reinterpret_cast<const uint4*>(V.child + 16ull * bi);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      uint4 t = __ldg(ct + k);
      kid[4 * k] = t.x, kid[4 * k + 1] = t.y, kid[4 * k + 2] = t.z, kid[4 * k + 3] = t.w;
    }
#pragma unroll
    for (int k = 0; k < 16; k++) {  // sixteen independent byte loads
      uint32_t cl = kid[k] == NODE_EMPTY ? 0u : (uint32_t)V.ref_len[kid[k]];
      rem |= (kid[k] == NODE_EMPTY ? 0u : 1u) << k;
      hmask |= (cl == 32 ? 1u : 0u) << k;
      payload += kid[k] == NODE_EMPTY ? 1u : (cl == 32 ? 33u : cl);
    }
    nunit = 1 + ((uint32_t)__popc(rem) + 2) / 3;
    total = len_prefix_size(payload) + payload;
  }
  Stage<B> s;
  s.init(smem);
  uint64_t a[25];
#pragma unroll
  for (int k = 0; k < 25; k++) a[k] = 0;
  uint4 rx = make_uint4(0, 0, 0, 0), ry = rx;  // ref of the message just finished
  uint32_t rlen = 0;
  for (;;) {
    bool permute = false, last = false;
    if (busy) {
      if (phase == 0) {
        while (s.bytes() < 136 && unit < nunit) {
          if (unit == 0) {
            emit_len_prefix(s, payload, 0xc0, 0xf7);
          } else {
            // three children per unit, walked in compact order so that the lanes of a warp emit their
            // j-th child together whatever slots the children sit in.  The child table was written by
            // earlier launches: re-reading an id is an L1 / L2 hit.
            uint32_t nib[3], cid[3];
            uint4 x[3], y[3];
#pragma unroll
            for (int t = 0; t < 3; t++) {
              nib[t] = rem ? (uint32_t)__ffs(rem) - 1 : 16u;
              rem &= rem - 1;
              cid[t] = nib[t] < 16 ? __ldg(V.child + 16ull * bi + nib[t]) : 0u;
            }
#pragma unroll
            for (int t = 0; t < 3; t++) {
              if (nib[t] < 16) {
                const uint4* q = reinterpret_cast<const uint4*>(V.ref + 32ull * cid[t]);
                x[t] = __ldcg(q), y[t] = __ldcg(q + 1);
              }
            }
#pragma unroll
            for (int t = 0; t < 3; t++) {
              if (nib[t] < 16) {
                emit_empty_run(s, nib[t] - next_slot);
                emit_ref(s, x[t], y[t], ((hmask >> nib[t]) & 1) ? 32u : (uint32_t)V.ref_len[cid[t]]);
                next_slot = nib[t] + 1;
              }
            }
            if (rem == 0) emit_empty_run(s, 17 - next_slot);  // trailing empty slots and the empty value
          }
          unit++;
        }
      }
      const bool final_msg = (phase == 1) || ext_len == 0;
      if (total < 32 && !(final_msg && is_root)) {
        inline_ref_words(s, total, rx, ry);
        rlen = total;
      } else {
        // (total < 32 here only for the root's last message; a sub-trie's parent would embed it, not its hash)
        if (total < 32 && V.base_depth > 0) atomicOr(V.flags, BUILD_F_SHORT_TOP);
        last = s.bytes() < 136;
        if (last) s.pad();
        absorb_stage<B>(a, s);
        permute = true;
      }
    }
    if (!__any_sync(FULL, busy)) break;
    if (__any_sync(FULL, permute)) keccak_f1600(a);
    if (busy) {
      bool msg_done = !permute;
      if (permute) {
        perms++;
        if (last) {
          digest_words(a, rx, ry);
          rlen = 32;
          hashed++;
          enc_bytes += total;
          msg_done = true;
        } else {
          s.consume_block();
        }
      }
      if (msg_done) {
        if (INNER && phase == 0) {
          uint4* o = reinterpret_cast<uint4*>(V.inner_ref + 32ull * bi);
          o[0] = rx, o[1] = ry;
          V.inner_ref_len[bi] = (uint8_t)rlen;
        }
        if (phase == 1 || ext_len == 0) {
          busy = false;
        } else {
          // the extension node above this branch: rlp[ hex_prefix(nibbles, false), ref ]
          phase = 1;
#pragma unroll
          for (int k = 0; k < 25; k++) a[k] = 0;
          s.init(smem);
          payload = hex_prefix_str_size(ext_len) + (rlen == 32 ? 33u : rlen);
          total = len_prefix_size(payload) + payload;
          emit_len_prefix(s, payload, 0xc0, 0xf7);
          emit_hex_prefix_str(s, V.keys + 32ull * V.rep[bi], es, ext_len, 0);
          emit_ref(s, rx, ry, rlen);
        }
      }
    }
  }
  if (slot < end) {
    uint4* o = reinterpret_cast<uint4*>(V.ref + 32ull * id);
    o[0] = rx, o[1] = ry;
    V.ref_len[id] = (uint8_t)rlen;
    if (is_root) {
      uint4* ro = reinterpret_cast<uint4*>(V.root_out);
      ro[0] = rx, ro[1] = ry;
    }
  }
  add_counters(V.counters, hashed, perms, enc_bytes);
}

// ------------------------------------------------------------------ launchers -----------------

static constexpr int HB = 128;
static inline uint32_t cdiv(uint64_t a, uint32_t b) { return (uint32_t)((a + b - 1) / b); }

void launch_lcp(const uint8_t* keys, uint32_t n, int8_t* L, uint32_t* flags, cudaStream_t st, int base_depth) {
  lcp_kernel<<<cdiv((uint64_t)n + 1, 256), 256, 0, st>>>(keys, n, L, flags, base_depth - 1);
}
void launch_min64(const int8_t* in, uint32_t n_in, int8_t* out, uint32_t n_out, cudaStream_t st) {
  min64_kernel<<<cdiv(n_out, 256), 256, 0, st>>>(in, n_in, out, n_out);
}
void launch_leaders(const int8_t* L, const int8_t* m1, const int8_t* m2, const int8_t* m3, uint32_t n, uint32_t* link_a, uint32_t* link_b,
                    uint32_t* flag, cudaStream_t st) {
  Pyramid P{L, m1, m2, m3};
  uint32_t g = cdiv((uint64_t)n + 1, 256);
  link_kernel<<<g, 256, 0, st>>>(P, n, link_a);
  // a branch has at most 16 children, so a chain has at most 15 links: 4 doublings
  jump_kernel<<<g, 256, 0, st>>>(link_a, link_b, n + 1);
  jump_kernel<<<g, 256, 0, st>>>(link_b, link_a, n + 1);
  jump_kernel<<<g, 256, 0, st>>>(link_a, link_b, n + 1);
  jump_kernel<<<g, 256, 0, st>>>(link_b, link_a, n + 1);
  leader_flag_kernel<<<g, 256, 0, st>>>(link_a, n, flag);
}
void launch_branch_info(const BuildView& V, cudaStream_t st) {
  if (V.n < 2) return;
  branch_info_kernel<<<cdiv(V.n, 256), 256, 0, st>>>(V);
}
void launch_child_count(const uint32_t* leader, const uint32_t* bidx, uint32_t n, uint32_t* nchild, cudaStream_t st) {
  if (n < 2) return;
  child_count_kernel<<<cdiv(n, 256), 256, 0, st>>>(leader, bidx, n, nchild);
}
void launch_hash_sorted_leaves(const BuildView& V, cudaStream_t st) {
  if (!V.n) return;
  hash_sorted_leaves_kernel<HB><<<cdiv(V.n, HB), HB, 0, st>>>(V);
}
void launch_hash_listed_leaves(const BuildView& V, const uint32_t* list, uint32_t count, cudaStream_t st) {
  if (!count) return;
  hash_sorted_leaves_kernel<HB><<<cdiv(count, HB), HB, 0, st>>>(V, LeafList{list, count});
}
void launch_hash_branch_level(const BuildView& V, const uint32_t* order, uint32_t begin, uint32_t end, cudaStream_t st) {
  if (end <= begin) return;
  if (V.inner_ref)
    hash_branch_level_kernel<HB, true><<<cdiv(end - begin, HB), HB, 0, st>>>(V, order, begin, end);
  else
    hash_branch_level_kernel<HB, false><<<cdiv(end - begin, HB), HB, 0, st>>>(V, order, begin, end);
}

}  // namespace ppd
