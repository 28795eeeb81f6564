// ppd_subset.cu — create_trie_subset (decoding.rs:551-602, eth_trie_utils trie_subsets.rs) of a trie the builder of
// ppd_build.cu has just built and hashed, for a set of query keys, serialised in the pre-order Node form of
// include/ppd_flat.h.  Runs within the same call as the builder, on its arrays (BuildView).
//
// Stages:
//   mark   one thread per query walks from the root (extension nibbles against rep's key, then child[b][nibble]) and
//          sets the bits of every node it reaches: a leaf, a branch, or only the extension above a branch when the key
//          leaves the trie inside it.  A branch touched for the first time is appended to its depth's bucket (a query
//          touches at most one branch per depth).  Repeated queries set the same bits.
//   size   one launch per depth, deepest first, a half-warp per touched branch (lane k: slot k): its size in the output
//   root   the root's offset (0) and the total; a root that is not a touched branch is written here
//   emit   one launch per depth, root down: each touched branch writes its extension, its kind byte, every child that
//          is not a touched branch, and the empty value, and hands each touched branch child its offset.
// A child that is not touched is HASH(ref) when its ref is 32 bytes; otherwise it encodes to fewer than 32 bytes and
// is written out whole (put_inline).  Sizes and bytes come from the same functions (W = false / true).
//
// Node form: EMPTY = 1 byte, HASH = 33, LEAF = 2 + nibbles + 4 + value, EXTENSION = 2 + nibbles + child,
// BRANCH = 1 + 16 children + 4 (value_len; a trie of 32-byte keys has no branch values).
#include <cstdint>

#include "../../include/ppd_flat.h"
#include "ppd_kernels.h"

namespace ppd {

static constexpr uint32_t FULL = 0xffffffffu;

__device__ __forceinline__ bool bit(const uint32_t* bits, uint64_t i) { return (__ldg(bits + (i >> 5)) >> (i & 31)) & 1u; }
// sets bit i; true when this call set it
__device__ __forceinline__ bool set_bit(uint32_t* bits, uint64_t i) {
  const uint32_t m = 1u << (i & 31);
  if (*(volatile uint32_t*)(bits + (i >> 5)) & m) return false;  // the top of the trie: every walk passes there
  return !(atomicOr(bits + (i >> 5), m) & m);
}

__device__ __forceinline__ uint32_t key_nibble(const uint8_t* key, uint32_t k) {
  const uint32_t b = key[k >> 1];
  return (k & 1) ? (b & 15u) : (b >> 4);
}

template <bool W>
__device__ __forceinline__ void put_u32(uint8_t* out, uint32_t v) {
  if (W)
    for (int k = 0; k < 4; k++) out[k] = (uint8_t)(v >> (8 * k));
}

template <bool W>
__device__ __forceinline__ uint64_t put_hash(const uint8_t* ref32, uint8_t* out) {
  if (W) {
    const uint4* q = reinterpret_cast<const uint4*>(ref32);
    const uint4 a = q[0], b = q[1];
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    out[0] = PPD_NODE_HASH;
#pragma unroll
    for (int k = 0; k < 32; k++) out[1 + k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
  }
  return 33;
}

// leaf i, spelling its key from nibble nib_from on
template <bool W>
__device__ __forceinline__ uint64_t put_leaf(const SubsetView& S, uint32_t i, uint32_t nib_from, uint8_t* out) {
  const uint64_t vo = S.val_off[i];
  const uint32_t vlen = (uint32_t)(S.val_off[i + 1] - vo), nn = 64 - nib_from;
  if (W) {
    const uint8_t* key = S.keys + 32ull * i;
    out[0] = PPD_NODE_LEAF, out[1] = (uint8_t)nn;
    for (uint32_t k = 0; k < nn; k++) out[2 + k] = (uint8_t)key_nibble(key, nib_from + k);
    put_u32<W>(out + 2 + nn, vlen);
    const uint8_t* v = S.vals + vo;
    for (uint32_t k = 0; k < vlen; k++) out[6 + nn + k] = v[k];
  }
  return 6ull + nn + vlen;
}

// the extension above branch b, without its child
template <bool W>
__device__ __forceinline__ uint64_t put_ext(const SubsetView& S, uint32_t b, uint8_t* out) {
  const uint32_t es = S.ext_start[b], d = S.depth[b];
  if (W) {
    const uint8_t* key = S.keys + 32ull * S.rep[b];
    out[0] = PPD_NODE_EXTENSION, out[1] = (uint8_t)(d - es);
    for (uint32_t k = es; k < d; k++) out[2 + k - es] = (uint8_t)key_nibble(key, k);
  }
  return 2 + d - es;
}

// Node c (a leaf, or branch c - N with its extension when with_ext) and everything below it, expanded: a node that
// encodes to fewer than 32 bytes, whose children are embedded raw too.  Such a subtree holds at most one branch below
// another (a branch encodes to 17 bytes or more), so a stack of four branches never fills up.
static constexpr int INLINE_STACK = 4;
template <bool W>
__device__ __forceinline__ uint64_t put_inline(const SubsetView& S, uint32_t c, bool with_ext, uint32_t nib_from, uint8_t* out) {
  uint32_t sb[INLINE_STACK], ss[INLINE_STACK];
  int sp = 0;
  uint64_t pos = 0;
  for (;;) {
    if (c < S.n) {
      pos += put_leaf<W>(S, c, nib_from, out + pos);
    } else {
      const uint32_t b = c - S.n;
      if (with_ext) pos += put_ext<W>(S, b, out + pos);
      if (sp == INLINE_STACK) {
        atomicOr(S.flags, SUBSET_F_DEEP);
        return pos;
      }
      if (W) out[pos] = PPD_NODE_BRANCH;
      pos++;
      sb[sp] = b, ss[sp] = 0, sp++;
    }
    for (;;) {  // the next node in pre-order
      if (sp == 0) return pos;
      const uint32_t b = sb[sp - 1], k = ss[sp - 1];
      if (k == 16) {
        put_u32<W>(out + pos, 0);
        pos += 4;
        sp--;
        continue;
      }
      ss[sp - 1] = k + 1;
      c = S.child[16ull * b + k];
      if (c == NODE_EMPTY) {
        if (W) out[pos] = PPD_NODE_EMPTY;
        pos++;
        continue;
      }
      nib_from = S.depth[b] + 1, with_ext = true;
      break;
    }
  }
}

// Child c of a branch (nib_from = its depth + 1), or the root (nib_from = 0).  A touched branch is written by the emit
// pass at the offset its parent gives it: here it only reports its size.
template <bool W>
__device__ __forceinline__ uint64_t put_child(const SubsetView& S, uint32_t c, uint32_t nib_from, uint8_t* out) {
  if (c == NODE_EMPTY) {
    if (W) out[0] = PPD_NODE_EMPTY;
    return 1;
  }
  const bool touched = bit(S.bits, c);
  if (c < S.n) return touched || S.ref_len[c] < 32 ? put_leaf<W>(S, c, nib_from, out) : put_hash<W>(S.ref + 32ull * c, out);
  const uint32_t b = c - S.n;
  if (touched) return S.so[b];
  if (bit(S.bits, (uint64_t)S.n + S.nb + b)) {  // a key left the trie inside the extension above b: b is embedded below it
    const uint64_t h = put_ext<W>(S, b, out);
    return h + (S.inner_ref_len[b] < 32 ? put_inline<W>(S, c, false, 0, out + h) : put_hash<W>(S.inner_ref + 32ull * b, out + h));
  }
  return S.ref_len[c] < 32 ? put_inline<W>(S, c, true, nib_from, out) : put_hash<W>(S.ref + 32ull * c, out);
}

// ------------------------------------------------------------------ mark ------------------------------------------------
__global__ void __launch_bounds__(256) subset_mark_kernel(SubsetView S, const uint8_t* __restrict__ queries32, uint32_t m) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
  bool live = i < m;
  uint32_t q[8];  // the query as big-endian words
  if (live) {
    const uint4* p = reinterpret_cast<const uint4*>(queries32 + 32ull * i);
    const uint4 a = __ldg(p), b = __ldg(p + 1);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int k = 0; k < 8; k++) q[k] = __byte_perm(w[k], 0, 0x0123);
  }
  uint32_t id = live ? *S.root_id : 0u;
  // warp-synchronous: every lane runs every round, so that lanes appending to the same depth take one atomic together
  for (;;) {
    bool append = false;
    uint32_t d = 0, b = 0;
    if (live) {
      if (id < S.n) {
        set_bit(S.bits, id);  // a leaf: the walk ends here, whatever its key
        live = false;
      } else {
        b = id - S.n;
        d = S.depth[b];
        const uint32_t es = S.ext_start[b];
        if (es < d) {
          set_bit(S.bits, (uint64_t)S.n + S.nb + b);
          // rep's key and the query agree on the nibbles above es (the walk took them): compare the extension's
          const uint4* p = reinterpret_cast<const uint4*>(S.keys + 32ull * S.rep[b]);
          const uint4 x = __ldg(p), y = __ldg(p + 1);
          const uint32_t r[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
          uint32_t lcp = 64;
#pragma unroll
          for (int k = 7; k >= 0; k--) {
            const uint32_t diff = __byte_perm(r[k], 0, 0x0123) ^ q[k];
            if (diff) lcp = 8 * k + (__clz(diff) >> 2);
          }
          if (lcp < d) live = false;  // the key leaves the trie inside the extension
        }
        if (live) {
          append = set_bit(S.bits, id);
          uint32_t w = 0;
#pragma unroll
          for (int k = 0; k < 8; k++) w = (k == (int)(d >> 3)) ? q[k] : w;
          const uint32_t c = S.child[16ull * b + ((w >> (28 - 4 * (d & 7))) & 15u)];
          if (c == NODE_EMPTY)
            live = false;  // an empty slot: the branch proves the key absent
          else
            id = c;
        }
      }
    }
    const uint32_t peers = __match_any_sync(FULL, append ? d : 0xffffffffu);
    const uint32_t leader = __ffs(peers) - 1;
    uint32_t slot = 0;
    if (append && lane == leader) slot = atomicAdd(S.count + d, (uint32_t)__popc(peers));
    slot = __shfl_sync(FULL, slot, leader) + __popc(peers & ((1u << lane) - 1));
    if (append && S.base[d] + slot < S.base[d + 1]) S.list[S.base[d] + slot] = b;
    if (!__any_sync(FULL, live)) break;
  }
}

// ------------------------------------------------------------------ size and emit ---------------------------------------
// Half-warp h of the launch takes touched branch list[base[d] + h]; lane k of it takes slot k.
__device__ __forceinline__ uint32_t half_scan(uint32_t lane16, uint64_t& v) {  // inclusive scan over the 16 lanes
#pragma unroll
  for (int s = 1; s < 16; s <<= 1) {
    const uint64_t u = __shfl_up_sync(FULL, v, s, 16);
    if (lane16 >= (uint32_t)s) v += u;
  }
  return lane16;
}

__global__ void __launch_bounds__(256) subset_size_kernel(SubsetView S, uint32_t d, uint32_t count) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, h = t >> 4, k = t & 15;
  const bool ok = h < count;
  uint32_t b = 0;
  uint64_t v = 0;
  if (ok) {
    b = S.list[S.base[d] + h];
    v = put_child<false>(S, S.child[16ull * b + k], d + 1, nullptr);
  }
#pragma unroll
  for (int s = 8; s >= 1; s >>= 1) v += __shfl_xor_sync(FULL, v, s, 16);
  if (ok && k == 0) {
    const uint32_t es = S.ext_start[b];
    S.so[b] = v + 5 + (es < d ? 2 + d - es : 0);  // + kind byte and value_len, + the extension
  }
}

__global__ void subset_root_kernel(SubsetView S, uint8_t* out, bool emit) {
  const uint32_t r = *S.root_id;
  if (r >= S.n && bit(S.bits, r)) {  // a touched root branch writes itself in the emit pass, at offset 0
    if (!emit) {
      *S.total = S.so[r - S.n];
      S.so[r - S.n] = 0;
    }
    return;
  }
  if (emit)
    put_child<true>(S, r, 0, out);
  else
    *S.total = put_child<false>(S, r, 0, nullptr);
}

__global__ void __launch_bounds__(256) subset_emit_kernel(SubsetView S, uint32_t d, uint32_t count, uint8_t* __restrict__ out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, h = t >> 4, k = t & 15;
  const bool ok = h < count;
  uint32_t b = 0, c = NODE_EMPTY;
  uint64_t v = 0;
  if (ok) {
    b = S.list[S.base[d] + h];
    c = S.child[16ull * b + k];
    v = put_child<false>(S, c, d + 1, nullptr);
  }
  uint64_t incl = v;
  half_scan(k, incl);
  const uint64_t children = __shfl_sync(FULL, incl, 15, 16);
  if (!ok) return;
  const uint32_t es = S.ext_start[b];
  const uint64_t o = S.so[b], head = 1 + (es < d ? 2 + d - es : 0);
  const uint64_t at = o + head + incl - v;
  if (c != NODE_EMPTY && c >= S.n && bit(S.bits, c))
    S.so[c - S.n] = at;  // a touched branch child: its offset replaces its size
  else
    put_child<true>(S, c, d + 1, out + at);
  if (k == 0) {
    if (es < d) put_ext<true>(S, b, out + o);
    out[o + head - 1] = PPD_NODE_BRANCH;
  }
  if (k == 15) put_u32<true>(out + o + head + children, 0);
}

// ------------------------------------------------------------------ launchers -------------------------------------------
static inline uint32_t cdiv(uint64_t a, uint32_t b) { return (uint32_t)((a + b - 1) / b); }

void launch_subset_mark(const SubsetView& S, const uint8_t* queries32, uint32_t m, cudaStream_t st) {
  if (!m) return;
  subset_mark_kernel<<<cdiv(m, 256), 256, 0, st>>>(S, queries32, m);
}
void launch_subset_size(const SubsetView& S, uint32_t d, uint32_t count, cudaStream_t st) {
  if (!count) return;
  subset_size_kernel<<<cdiv(16ull * count, 256), 256, 0, st>>>(S, d, count);
}
void launch_subset_root(const SubsetView& S, uint8_t* out, bool emit, cudaStream_t st) { subset_root_kernel<<<1, 1, 0, st>>>(S, out, emit); }
void launch_subset_emit(const SubsetView& S, uint32_t d, uint32_t count, uint8_t* out, cudaStream_t st) {
  if (!count) return;
  subset_emit_kernel<<<cdiv(16ull * count, 256), 256, 0, st>>>(S, d, count, out);
}

}  // namespace ppd
