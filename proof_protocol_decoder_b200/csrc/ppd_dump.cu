// ppd_dump.cu — serialising the per-txn sub-tries (IrDump "Trie" blobs, include/ppd_flat.h) ON THE GPU.
//
// Replaces the host walk that cut every txn's minimal sub-tries out of the hashed arena
// (create_trie_subset, decoding.rs:551-602: keep every node on the path of an accessed key, replace
// every untouched subtree by Hash(subtree hash)).  After the sweep the arena, the witness hashes and
// every ref are resident in HBM, so cutting a subset is a gather: the host only uploads, per IR, the
// ids of the nodes its keys touched and the order of its tries; the device
//   1. ir_size_kernel  (one CTA per IR): de-duplicates the touched ids in a shared-memory hash set,
//      computes every touched node's serialised size bottom-up (children that are touched are looked
//      up in the set, all others are 1 byte (empty) or 33 bytes (hash)), lays the IR's segments
//      (host literals and tries) out, and assigns every touched node its byte offset top-down;
//   2. ir_emit_kernel  (one CTA per IR): every touched node writes its own bytes at its offset.
// The IR's literal bytes (counters, signed txn, code map ...) are written by the host into the holes.
// An IR the kernels cannot lay out (more unique touched nodes than the set holds, a node shared by two
// tries of the IR, an untouched child whose encoding is shorter than 32 bytes, which the subset keeps
// expanded) is flagged and serialised by the host instead.
#include <cstddef>
#include <cstdint>

#include "../../include/ppd_flat.h"
#include "arena.h"
#include "ppd_kernels.h"
#include "scan.cuh"

namespace ppd {

namespace {

constexpr uint32_t HASH_ID_BASE = 0x80000000u;
constexpr uint32_t SET_CAP = 8192, MAX_UNIQ = 4096, NOT_FOUND = 0xffffffffu, UNSET = 0xffffffffu;
#ifndef PPD_DUMP_THREADS
#define PPD_DUMP_THREADS 1024
#endif
constexpr int DUMP_THREADS = PPD_DUMP_THREADS;

// The set of an IR's touched nodes.  For an ordinary IR (at most MAX_UNIQ distinct touched nodes) everything lives in
// shared memory; for a big one (a txn that writes tens of thousands of slots: config 3) the table and the per-node
// arrays are in HBM (table: the block's scratch; arrays: the plan's u_node / u_size / u_off themselves).
struct SharedSet {
  uint32_t key[SET_CAP];   // node id or NODE_EMPTY
  uint32_t slot[SET_CAP];  // index into the u_* arrays
  uint32_t u_node[MAX_UNIQ], u_size[MAX_UNIQ], u_off[MAX_UNIQ];
  uint32_t u_par[MAX_UNIQ];  // index of the touched node's touched parent (ir_size_kernel)
};
struct Set {
  uint32_t *key, *slot, *u_node, *u_size, *u_off, *u_par;
  uint32_t shift, mask, max_uniq;
  uint32_t n_uniq, n_done, flag;  // (this struct lives in shared memory)
};

__device__ __forceinline__ uint32_t hash_slot(const Set& s, uint32_t id) { return (id * 2654435761u) >> s.shift; }

__device__ __forceinline__ uint32_t set_find(const Set& s, uint32_t id) {
  uint32_t h = hash_slot(s, id);
  for (;;) {
    uint32_t k = s.key[h];
    if (k == id) return s.slot[h];
    if (k == NODE_EMPTY) return NOT_FOUND;
    h = (h + 1) & s.mask;
  }
}

// points the set at shared memory, or at the IR's region of the big-IR scratch
__device__ void set_bind(Set& s, SharedSet& sm, const IrDumpPlanView& P, uint32_t ir, uint32_t tb) {
  if (threadIdx.x == 0) {
    const uint64_t big = P.big_off ? P.big_off[ir] : ~0ull;
    if (big == ~0ull) {
      s.key = sm.key, s.slot = sm.slot, s.u_node = sm.u_node, s.u_size = sm.u_size, s.u_off = sm.u_off, s.u_par = sm.u_par;
      s.mask = SET_CAP - 1, s.shift = 19, s.max_uniq = MAX_UNIQ;
    } else {
      const uint32_t cap = P.big_cap[ir];  // a power of two >= 2 x the IR's touched slots
      s.key = P.big_scratch + big, s.slot = s.key + cap, s.u_par = s.slot + cap;  // (3 x cap words per big IR)
      s.u_node = P.u_node + tb, s.u_size = P.u_size + tb, s.u_off = P.u_off + tb;
      s.mask = cap - 1, s.shift = 32 - (31 - __clz(cap)), s.max_uniq = cap / 2;
    }
  }
  __syncthreads();
}

__device__ __forceinline__ bool is_hash_id(uint32_t id) { return id >= HASH_ID_BASE && id != NODE_EMPTY; }
__device__ __forceinline__ uint32_t node_kind(const ArenaView& A, uint32_t id) { return A.nodes[id].w0 & 0xff; }

__device__ __forceinline__ uint32_t u256_sig(const uint8_t* be) {
  uint32_t i = 0;
  while (i < 32 && be[i] == 0) i++;
  return 32 - i;
}
__device__ __forceinline__ uint32_t u256_str_len(const uint8_t* be, uint32_t sig) { return sig == 0 ? 1u : (sig == 1 && be[31] < 0x80) ? 1u : 1u + sig; }
// rlp([nonce, balance, storage_root, code_hash]): always a long list (payload >= 68)
__device__ __forceinline__ uint32_t account_rlp_len(const AccountRec& r) {
  return 2 + u256_str_len(r.nonce, u256_sig(r.nonce)) + u256_str_len(r.balance, u256_sig(r.balance)) + 66;
}

// serialised size of child `c` of a touched node: 1 (empty), 33 (hash), its own size when it is touched
// itself (UNSET while that is not known yet).  Sets *flag for an untouched child kept expanded (< 32 bytes).
__device__ __forceinline__ uint32_t child_size(const ArenaView& A, const Set& s, uint32_t c, uint32_t* flag) {
  if (c == NODE_EMPTY) return 1;
  if (is_hash_id(c)) return 33;
  uint32_t k = set_find(s, c);
  if (k != NOT_FOUND) return s.u_size[k];
  if (A.ref_len[c] != 32 && node_kind(A, c) != NK_ROOT) *flag = 1;
  return 33;
}

// size of node u given its children's sizes, or UNSET when a touched child is not sized yet
__device__ uint32_t node_size(const ArenaView& A, const Set& s, uint32_t u, uint32_t* flag) {
  const NodeRec r = A.nodes[u];
  const uint32_t kind = r.w0 & 0xff, nlen = (r.w0 >> 16) & 0xff;
  switch (kind) {
    case NK_LEAF:
      return 1 + 1 + nlen + 4 + r.a2;
    case NK_LEAF_ACCOUNT:
      return 1 + 1 + nlen + 4 + account_rlp_len(A.accounts[r.a1]);
    case NK_EXT: {
      uint32_t cs = child_size(A, s, r.a1, flag);
      return cs == UNSET ? UNSET : 1 + 1 + nlen + cs;
    }
    case NK_BRANCH: {
      const uint32_t mask = r.a1 & 0xffff, k = __popc(mask);
      uint32_t total = 1 + (16 - k) + 4;
      for (uint32_t j = 0; j < k; j++) {
        uint32_t cs = child_size(A, s, A.child_pool[r.a0 + j], flag);
        if (cs == UNSET) return UNSET;
        total += cs;
      }
      return total;
    }
    default:  // NK_ROOT is never inserted
      *flag = 1;
      return 33;
  }
}

__device__ void build_set(Set& s, const uint32_t* ids, uint32_t n, const ArenaView& A, bool dedupe) {
  for (uint32_t i = threadIdx.x; i <= s.mask; i += blockDim.x) s.key[i] = NODE_EMPTY;
  if (threadIdx.x == 0) s.n_uniq = 0, s.n_done = 0, s.flag = 0;
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
    uint32_t id = ids[i];
    if (id == NODE_EMPTY || is_hash_id(id)) continue;
    if (dedupe && node_kind(A, id) == NK_ROOT) continue;  // opaque: always emitted as a hash by its parent
    uint32_t h = hash_slot(s, id);
    for (;;) {
      uint32_t prev = atomicCAS(&s.key[h], NODE_EMPTY, id);
      if (prev == NODE_EMPTY) {
        uint32_t k = dedupe ? atomicAdd(&s.n_uniq, 1u) : i;
        if (k < s.max_uniq) {
          s.slot[h] = k;
          s.u_node[k] = id;
        } else {
          s.flag = 1;
          s.slot[h] = 0;
        }
        break;
      }
      if (prev == id) break;
      h = (h + 1) & s.mask;
    }
  }
  __syncthreads();
}

}  // namespace

// One CTA per IR.  Outputs: ir_size, ir_flag, ir_nuniq, and at [touched_begin[ir] + k] the k-th unique
// touched node, its size and its offset inside the IR; seg_off[s] for every segment.
__global__ void __launch_bounds__(DUMP_THREADS) ir_size_kernel(ArenaView A, IrDumpPlanView P) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ Set s;
  const uint32_t ir = blockIdx.x;
  const uint32_t tb = P.touched_begin[ir], tn = P.touched_begin[ir + 1] - tb;
  set_bind(s, *reinterpret_cast<SharedSet*>(smem_raw), P, ir, tb);
  build_set(s, P.touched + tb, tn, A, true);
  const uint32_t nu = min(s.n_uniq, s.max_uniq);
  constexpr uint32_t PLACED = 0x80000000u, NO_KIDS = 0x40000000u;
  for (uint32_t k = threadIdx.x; k < nu; k += blockDim.x) s.u_par[k] = UNSET;
  __syncthreads();
  // ---- pass 1 (the only one that waits for HBM): per touched node, the bytes that do not depend on other touched
  // nodes (its own fields, its untouched children: 1 byte empty, 33 hashed), how many touched children it has, and
  // every touched child's parent.  The touched nodes of a trie form a tree: sizes then flow up it in shared memory. ----
  {
    uint32_t local_flag = 0;
    for (uint32_t k = threadIdx.x; k < nu; k += blockDim.x) {
      const NodeRec r = A.nodes[s.u_node[k]];
      const uint32_t kind = r.w0 & 0xff, nlen = (r.w0 >> 16) & 0xff;
      uint32_t fixed = 0, pend = 0;
      auto child = [&](uint32_t c) {
        if (c == NODE_EMPTY) return 1u;
        if (is_hash_id(c)) return 33u;
        const uint32_t kc = set_find(s, c);
        if (kc != NOT_FOUND) {
          if (atomicCAS(&s.u_par[kc], UNSET, k) != UNSET) local_flag = 1;  // a node with two touched parents
          pend++;
          return 0u;
        }
        if (A.ref_len[c] != 32 && node_kind(A, c) != NK_ROOT) local_flag = 1;  // an untouched child the subset keeps expanded
        return 33u;
      };
      switch (kind) {
        case NK_LEAF:
          fixed = 1 + 1 + nlen + 4 + r.a2;
          break;
        case NK_LEAF_ACCOUNT:
          fixed = 1 + 1 + nlen + 4 + account_rlp_len(A.accounts[r.a1]);
          break;
        case NK_EXT:
          fixed = 1 + 1 + nlen + child(r.a1);
          break;
        case NK_BRANCH: {
          const uint32_t mask = r.a1 & 0xffff, nk = __popc(mask);
          uint32_t cid[16];
#pragma unroll
          for (uint32_t j = 0; j < 16; j++) cid[j] = j < nk ? A.child_pool[r.a0 + j] : NODE_EMPTY;  // (all in flight together)
          fixed = 1 + (16 - nk) + 4;
#pragma unroll
          for (uint32_t j = 0; j < 16; j++)
            if (j < nk) fixed += child(cid[j]);
          break;
        }
        default:  // NK_ROOT is never inserted
          local_flag = 1;
          fixed = 33;
      }
      s.u_size[k] = fixed;
      s.u_off[k] = pend ? pend : NO_KIDS;  // (until the segments are laid out: the touched children that have yet to report)
    }
    if (local_flag) s.flag = 1;
  }
  __syncthreads();
  // ---- sizes flow up: a node without touched children is final; it adds its size to its parent's, and whoever
  // reports last to a parent carries on from there ----
  for (uint32_t k = threadIdx.x; k < nu; k += blockDim.x) {
    if (s.u_off[k] != NO_KIDS) continue;  // (a parent's count may reach 0 while this loop runs: it is carried on by its last child)
    uint32_t cur = k;
    for (uint32_t guard = 0; guard < 128; guard++) {
      const uint32_t p = s.u_par[cur];
      if (p == UNSET) break;
      atomicAdd(&s.u_size[p], *reinterpret_cast<volatile uint32_t*>(&s.u_size[cur]));
      __threadfence_block();
      if (atomicSub(&s.u_off[p], 1u) != 1u) break;
      __threadfence_block();
      cur = p;
    }
  }
  __syncthreads();
  {
    uint32_t stuck = 0;
    for (uint32_t k = threadIdx.x; k < nu; k += blockDim.x) {
      stuck |= s.u_off[k] & ~NO_KIDS;
      s.u_off[k] = UNSET;
    }
    if (stuck) s.flag = 1;  // (a cycle of parents: not a trie)
  }
  __syncthreads();
  // ---- segments: literals and tries in output order.  Every segment's size in parallel, then a block-wide
  // exclusive scan in chunks of DUMP_THREADS (an IR of a mainnet-shaped block has ~250 segments) ----
  {
    __shared__ uint32_t scan_warp[DUMP_THREADS / 32];
    __shared__ uint32_t scan_carry;
    if (threadIdx.x == 0) scan_carry = 0;
    __syncthreads();
    const uint32_t sb = P.seg_begin[ir], se = P.seg_end ? P.seg_end[ir] : P.seg_begin[ir + 1];
    for (uint32_t q0 = sb; q0 < se; q0 += DUMP_THREADS) {
      const uint32_t q = q0 + threadIdx.x;
      uint32_t sz = 0, trie_slot = NOT_FOUND;
      if (q < se) {
        const uint32_t a = P.seg_a[q], b = P.seg_b[q];
        if (b == NODE_EMPTY) {
          sz = 1;
        } else if (b == IR_SEG_ROOT_ONLY) {
          // a trie of which only the root is kept (create_trie_subset with the key 0_u64, decoding.rs:466-471)
          if (a == NODE_EMPTY) {
            sz = 1;
          } else if (is_hash_id(a) || node_kind(A, a) == NK_ROOT) {
            sz = 33;
          } else {
            uint32_t fl = 0;
            sz = node_size(A, s, a, &fl);
            if (fl) s.flag = 1;
          }
        } else if (b >= IR_SEG_KIND_MIN) {
          sz = (b == IR_SEG_REF || b == IR_SEG_KEY32) ? 32u : a;
        } else if (is_hash_id(b)) {
          sz = 33;
        } else {
          sz = 33;
          const uint32_t k = set_find(s, b);
          if (k != NOT_FOUND) {
            trie_slot = k;
            sz = s.u_size[k];
          } else if (A.ref_len[b] != 32 && node_kind(A, b) != NK_ROOT) {
            s.flag = 1;
          }
        }
      }
      const uint32_t incl = warp_inclusive_scan(sz, threadIdx.x & 31);
      if ((threadIdx.x & 31) == 31) scan_warp[threadIdx.x >> 5] = incl;
      __syncthreads();
      uint32_t before = scan_carry;
      for (uint32_t w = 0; w < (threadIdx.x >> 5); w++) before += scan_warp[w];
      const uint32_t off = before + incl - sz;
      if (q < se) {
        P.seg_off[q] = off;
        if (trie_slot != NOT_FOUND && atomicCAS(&s.u_off[trie_slot], UNSET, off) != UNSET) s.flag = 1;  // a node that roots two tries of one IR
      }
      __syncthreads();
      if (threadIdx.x == DUMP_THREADS - 1) scan_carry = off + sz;
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      P.ir_size[ir] = scan_carry;
      s.n_done = 0;
    }
  }
  __syncthreads();
  // ---- offsets.  Pass 2 over the arena (warm): every touched node places its touched children RELATIVE to its own
  // first byte; then the offsets flow down the tree in shared memory (a trie's root got its offset from its segment) ----
  if (!s.flag) {
    for (uint32_t k = threadIdx.x; k < nu; k += blockDim.x) {
      const NodeRec r = A.nodes[s.u_node[k]];
      const uint32_t kind = r.w0 & 0xff, nlen = (r.w0 >> 16) & 0xff;
      if (kind == NK_EXT) {
        const uint32_t c = is_hash_id(r.a1) ? NOT_FOUND : set_find(s, r.a1);
        if (c != NOT_FOUND) {
          if (s.u_off[c] != UNSET) s.flag = 1;  // (also the root of a trie of this IR)
          s.u_off[c] = 2 + nlen;
        }
      } else if (kind == NK_BRANCH) {
        const uint32_t mask = r.a1 & 0xffff, nk = __popc(mask);
        uint32_t cid[16];
#pragma unroll
        for (uint32_t j = 0; j < 16; j++) cid[j] = j < nk ? A.child_pool[r.a0 + j] : NODE_EMPTY;
        uint32_t off = 1;
        for (uint32_t i = 0, j = 0; i < 16; i++) {
          if (!(mask & (1u << i))) {
            off += 1;
            continue;
          }
          uint32_t c_id = NODE_EMPTY;
#pragma unroll
          for (uint32_t z = 0; z < 16; z++)
            if (z == j) c_id = cid[z];
          j++;
          const uint32_t c = is_hash_id(c_id) ? NOT_FOUND : set_find(s, c_id);
          if (c != NOT_FOUND) {
            if (s.u_off[c] != UNSET) s.flag = 1;
            s.u_off[c] = off;
            off += s.u_size[c];
          } else {
            off += 33;
          }
        }
      }
    }
  }
  __syncthreads();
  for (int round = 0; round < 130; round++) {
    __syncthreads();
    if (s.flag || s.n_done >= nu) break;  // uniform: nothing writes between the barrier and this read
    __syncthreads();
    uint32_t progressed = 0;
    for (uint32_t k = threadIdx.x; k < nu; k += blockDim.x) {
      if (*reinterpret_cast<volatile uint32_t*>(&s.u_size[k]) & PLACED) continue;
      const uint32_t p = s.u_par[k];
      uint32_t off = *reinterpret_cast<volatile uint32_t*>(&s.u_off[k]);
      if (p != UNSET) {
        if (!(*reinterpret_cast<volatile uint32_t*>(&s.u_size[p]) & PLACED)) continue;
        __threadfence_block();
        off += *reinterpret_cast<volatile uint32_t*>(&s.u_off[p]);
      } else if (off == UNSET) {
        s.flag = 1;  // a touched node no trie of the IR reaches
        continue;
      }
      s.u_off[k] = off;
      __threadfence_block();
      atomicOr(&s.u_size[k], PLACED);
      progressed++;
    }
    if (progressed) atomicAdd(&s.n_done, progressed);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s.n_done < nu) s.flag = 1;  // a touched node no trie of the IR reaches
    P.ir_flag[ir] = s.flag;
    P.ir_nuniq[ir] = nu;
  }
  for (uint32_t k = threadIdx.x; k < nu; k += blockDim.x) {
    const uint32_t node = s.u_node[k], size = s.u_size[k] & 0x7fffffffu, off = s.u_off[k];  // (a big IR's arrays ARE the plan's)
    P.u_node[tb + k] = node;
    P.u_size[tb + k] = size;
    P.u_off[tb + k] = off;
  }
}

namespace {

// PPD_NODE_HASH || 32 bytes at an arbitrary destination alignment: the 33 bytes are laid out as nine little-endian
// words, the bytes up to the first 4-byte boundary and after the last one are stored one by one, everything in
// between as aligned words re-aligned with funnel shifts (8 word stores instead of 33 byte stores; hashed-out
// children are most of an IR's bytes).
__device__ __forceinline__ uint8_t* put_hash_regs(uint8_t* q, const uint4 x, const uint4 y) {
  const uint32_t w[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
  uint32_t S[10];
  S[0] = (uint32_t)PPD_NODE_HASH | (w[0] << 8);
#pragma unroll
  for (int k = 1; k < 8; k++) S[k] = __funnelshift_r(w[k - 1], w[k], 24);
  S[8] = w[7] >> 24;
  S[9] = 0;
  const uint32_t head = (4u - (uint32_t)(reinterpret_cast<uintptr_t>(q) & 3u)) & 3u;  // bytes before the first aligned word
  for (uint32_t i = 0; i < head; i++) q[i] = (uint8_t)(S[0] >> (8 * i));
  uint32_t* qw = reinterpret_cast<uint32_t*>(q + head);
  const uint32_t sh = 8 * head, nwords = (33u - head) >> 2;  // 8 when head == 0 or 1 ... 7 when head == 2 or 3 (then 2 or 1 tail bytes)
#pragma unroll
  for (int j = 0; j < 8; j++)
    if ((uint32_t)j < nwords) qw[j] = __funnelshift_r(S[j], S[j + 1], sh);
  const uint32_t done = head + 4 * nwords;
  for (uint32_t i = done; i < 33; i++) q[i] = (uint8_t)(S[i >> 2] >> (8 * (i & 3)));
  return q + 33;
}
__device__ __forceinline__ uint8_t* put_hash(uint8_t* q, const uint8_t* h32) {
  const uint4* src = reinterpret_cast<const uint4*>(h32);
  return put_hash_regs(q, __ldg(src), __ldg(src + 1));
}
__device__ __forceinline__ uint8_t* put_u32(uint8_t* q, uint32_t v) {
  q[0] = (uint8_t)v, q[1] = (uint8_t)(v >> 8), q[2] = (uint8_t)(v >> 16), q[3] = (uint8_t)(v >> 24);
  return q + 4;
}
__device__ __forceinline__ uint8_t* put_nibbles(uint8_t* q, const ArenaView& A, const NodeRec& r) {
  const uint32_t start = (r.w0 >> 8) & 0xff, n = (r.w0 >> 16) & 0xff;
  const uint8_t* key = A.key_pool + r.a0;
  *q++ = (uint8_t)n;
  for (uint32_t i = 0; i < n; i++) {
    uint32_t b = key[(start + i) >> 1];
    *q++ = (uint8_t)(((start + i) & 1) ? (b & 15) : (b >> 4));
  }
  return q;
}
__device__ __forceinline__ uint8_t* put_u256_str(uint8_t* q, const uint8_t* be) {
  uint32_t sig = u256_sig(be);
  if (sig == 0) {
    *q++ = 0x80;
    return q;
  }
  if (!(sig == 1 && be[31] < 0x80)) *q++ = (uint8_t)(0x80 + sig);
  for (uint32_t i = 32 - sig; i < 32; i++) *q++ = be[i];
  return q;
}
// the child of a touched node: skipped when it is touched itself (it writes its own bytes)
__device__ __forceinline__ uint8_t* put_child(uint8_t* q, const ArenaView& A, const Set& s, uint32_t c) {
  if (c == NODE_EMPTY) {
    *q++ = PPD_NODE_EMPTY;
    return q;
  }
  if (is_hash_id(c)) return put_hash(q, A.hash_pool + 32ull * (c - HASH_ID_BASE));
  uint32_t k = set_find(s, c);
  if (k != NOT_FOUND) return q + s.u_size[k];
  return put_hash(q, A.ref + 32ull * c);
}

}  // namespace

// the bytes of node u at q: its own fields, and every child that is not touched itself (touched ones write themselves)
__device__ void emit_node(const ArenaView& A, const Set& s, uint32_t u, uint8_t* q) {
  const NodeRec r = A.nodes[u];
  switch (r.w0 & 0xff) {
    case NK_LEAF: {
      *q++ = PPD_NODE_LEAF;
      q = put_nibbles(q, A, r);
      q = put_u32(q, r.a2);
      const uint8_t* v = A.val_pool + r.a1;
      for (uint32_t i = 0; i < r.a2; i++) q[i] = v[i];
      break;
    }
    case NK_LEAF_ACCOUNT: {
      const AccountRec& acc = A.accounts[r.a1];
      *q++ = PPD_NODE_LEAF;
      q = put_nibbles(q, A, r);
      uint32_t len = account_rlp_len(acc);
      q = put_u32(q, len);
      *q++ = 0xf8;
      *q++ = (uint8_t)(len - 2);
      q = put_u256_str(q, acc.nonce);
      q = put_u256_str(q, acc.balance);
      const uint8_t* sr = acc.storage_src == NODE_EMPTY ? acc.storage_root : A.ref + 32ull * acc.storage_src;
      *q++ = 0xa0;
      for (int i = 0; i < 32; i++) *q++ = sr[i];
      *q++ = 0xa0;
      for (int i = 0; i < 32; i++) *q++ = acc.code_hash[i];
      break;
    }
    case NK_EXT:
      *q++ = PPD_NODE_EXTENSION;
      q = put_nibbles(q, A, r);
      put_child(q, A, s, r.a1);
      break;
    case NK_BRANCH: {
      // Children that are not touched themselves are 33-byte hashes gathered from all over the ref / hash pools: the
      // child ids are loaded together, then the hashes four children at a time (eight 16-byte loads in flight), so a
      // branch costs six round trips to memory instead of two per child.
      *q++ = PPD_NODE_BRANCH;
      const uint32_t mask = r.a1 & 0xffff, nk = __popc(mask);
      uint32_t cid[16];
#pragma unroll
      for (uint32_t j = 0; j < 16; j++) cid[j] = j < nk ? A.child_pool[r.a0 + j] : NODE_EMPTY;
      uint32_t m = mask;
      int prev_slot = -1;
#pragma unroll
      for (uint32_t g = 0; g < 16; g += 4) {
        if (g >= nk) break;
        const uint4* src[4];
        uint32_t skip[4];
        uint4 x[4], y[4];
#pragma unroll
        for (uint32_t z = 0; z < 4; z++) {
          const uint32_t c = cid[g + z];
          src[z] = nullptr, skip[z] = 0;
          if (g + z >= nk) continue;
          if (c == NODE_EMPTY) {
            skip[z] = NOT_FOUND;  // (not in a compact child row; sized as one byte by ir_size_kernel)
          } else if (is_hash_id(c)) {
            src[z] = reinterpret_cast<const uint4*>(A.hash_pool + 32ull * (c - HASH_ID_BASE));
          } else {
            const uint32_t k = set_find(s, c);
            if (k != NOT_FOUND)
              skip[z] = s.u_size[k];  // touched itself: it writes its own bytes
            else
              src[z] = reinterpret_cast<const uint4*>(A.ref + 32ull * c);
          }
        }
#pragma unroll
        for (uint32_t z = 0; z < 4; z++)
          if (src[z]) x[z] = __ldg(src[z]), y[z] = __ldg(src[z] + 1);
#pragma unroll
        for (uint32_t z = 0; z < 4; z++) {
          if (g + z >= nk) continue;
          const int slot = __ffs((int)m) - 1;
          m &= m - 1;
          for (int e = prev_slot + 1; e < slot; e++) *q++ = PPD_NODE_EMPTY;
          prev_slot = slot;
          if (src[z])
            q = put_hash_regs(q, x[z], y[z]);
          else if (skip[z] == NOT_FOUND)
            *q++ = PPD_NODE_EMPTY;
          else
            q += skip[z];
        }
      }
      for (int e = prev_slot + 1; e < 16; e++) *q++ = PPD_NODE_EMPTY;
      put_u32(q, 0);
      break;
    }
    default:
      break;
  }
}

// One CTA per IR: every unique touched node writes its own bytes at out + ir_base[ir] + its offset.
__global__ void __launch_bounds__(DUMP_THREADS) ir_emit_kernel(ArenaView A, IrDumpPlanView P, uint8_t* __restrict__ out) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ Set s;
  const uint32_t ir = blockIdx.x;
  if (P.ir_flag[ir]) return;  // serialised by the host
  const uint32_t tb = P.touched_begin[ir], nu = P.ir_nuniq[ir];
  set_bind(s, *reinterpret_cast<SharedSet*>(smem_raw), P, ir, tb);
  if (s.u_node != P.u_node + tb) {  // an ordinary IR: the set again in shared memory (a big IR's table is still in HBM)
    build_set(s, P.u_node + tb, nu, A, false);
    for (uint32_t k = threadIdx.x; k < nu; k += blockDim.x) s.u_size[k] = P.u_size[tb + k], s.u_off[k] = P.u_off[tb + k];
  }
  __syncthreads();
  uint8_t* base = out + P.ir_base[ir];
  for (uint32_t k = threadIdx.x; k < nu; k += blockDim.x) emit_node(A, s, s.u_node[k], base + s.u_off[k]);
  // the other segments: untouched tries (a storage trie nobody reads: its root as a hash, or empty), roots, hashed
  // addresses, and the literal bytes that are resident in HBM (FlatBlock ranges, the uploaded literal pool)
  const uint32_t sb = P.seg_begin[ir], se = P.seg_end ? P.seg_end[ir] : P.seg_begin[ir + 1];
  for (uint32_t qi = sb + threadIdx.x; qi < se; qi += blockDim.x) {
    const uint32_t b = P.seg_b[qi];
    if (b == IR_SEG_LITERAL) continue;
    uint8_t* q = base + P.seg_off[qi];
    if (b == IR_SEG_REF || b == IR_SEG_KEY32) {
      const uint8_t* r = b == IR_SEG_REF ? A.ref + 32ull * P.seg_a[qi] : A.key_pool + P.seg_a[qi];
      for (int i = 0; i < 32; i++) q[i] = r[i];
      continue;
    }
    if (b == IR_SEG_ROOT_ONLY) {
      const uint32_t a = P.seg_a[qi];
      if (a == NODE_EMPTY)
        *q = PPD_NODE_EMPTY;
      else if (is_hash_id(a))
        put_hash(q, A.hash_pool + 32ull * (a - HASH_ID_BASE));
      else if (node_kind(A, a) == NK_ROOT)
        put_hash(q, A.ref + 32ull * a);
      else
        emit_node(A, s, a, q);
      continue;
    }
    if (b == IR_SEG_FLAT || b == IR_SEG_LIT_DEV) {
      const uint32_t len = P.seg_a[qi];
      if (len > 96) continue;  // long ones: the whole block copies them below
      const uint8_t* src = (b == IR_SEG_FLAT ? P.flat : P.lit) + P.seg_c[qi];
      for (uint32_t i = 0; i < len; i++) q[i] = src[i];
      continue;
    }
    if (b == NODE_EMPTY)
      *q = PPD_NODE_EMPTY;
    else if (is_hash_id(b))
      put_hash(q, A.hash_pool + 32ull * (b - HASH_ID_BASE));
    else if (set_find(s, b) == NOT_FOUND)
      put_hash(q, A.ref + 32ull * b);
  }
  if (P.seg_c) {
    for (uint32_t qi = sb; qi < se; qi++) {
      const uint32_t b = P.seg_b[qi];
      if (b != IR_SEG_FLAT && b != IR_SEG_LIT_DEV) continue;
      const uint32_t len = P.seg_a[qi];
      if (len <= 96) continue;
      const uint8_t* src = (b == IR_SEG_FLAT ? P.flat : P.lit) + P.seg_c[qi];
      uint8_t* q = base + P.seg_off[qi];
      for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) q[i] = src[i];
    }
  }
}

size_t ir_dump_smem_bytes() { return sizeof(SharedSet); }

void launch_ir_size(const ArenaView& A, const IrDumpPlanView& P, uint32_t n_ir, cudaStream_t st) {
  if (!n_ir) return;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(ir_size_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SharedSet));
    cudaFuncSetAttribute(ir_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SharedSet));
    attr = true;
  }
  ir_size_kernel<<<n_ir, DUMP_THREADS, sizeof(SharedSet), st>>>(A, P);
}
void launch_ir_emit(const ArenaView& A, const IrDumpPlanView& P, uint32_t n_ir, uint8_t* out, cudaStream_t st) {
  if (!n_ir) return;
  ir_emit_kernel<<<n_ir, DUMP_THREADS, offsetof(SharedSet, u_par), st>>>(A, P, out);  // (no parents there: two thread blocks per SM)
}

}  // namespace ppd
