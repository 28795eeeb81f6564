// ppd_kernels.cu — sm_100a kernels of the hot path.
//
//   keccak256_batch_kernel   utils.rs:11-13 `hash` over a batch of messages (account addresses,
//                            storage slots, contract code: processed_block_trace.rs:219,234,277;
//                            decoding.rs:235,411; compact_to_partial_trie.rs:87,147)
//   hash_level_kernel        one level of the bottom-up root computation: per node, RLP-encode it
//                            straight into a Keccak sponge (eth_trie_utils Node::hash_intern,
//                            SURVEY.md 3.3) and store its "ref" for the parent level.
//
// Both are thread-per-sponge: the state stays in registers, the 136-byte rate block is staged in
// a conflict-free shared-memory slice owned by the thread (keccak.cuh).  Each kernel has exactly
// one keccak_f1600 site inside a loop over rate blocks: filling the next block is cheap and may
// diverge, the permutation (98 % of the instructions) is executed convergently by the warp.
#include <cstdint>

#include "arena.h"
#include "encode.cuh"
#include "keccak.cuh"
#include "ppd_kernels.h"

namespace ppd {

using namespace enc;

static constexpr uint32_t FULL = 0xffffffffu;

// A child id is an arena node or, from HASH_ID_BASE up, an entry of hash_pool (a hashed-out subtree of
// the witness: its ref is the 32 bytes themselves, nothing is computed for it).
static constexpr uint32_t HASH_ID_BASE = 0x80000000u;
__device__ __forceinline__ const uint8_t* ref_ptr(const ArenaView& A, uint32_t id) {
  return id >= HASH_ID_BASE ? A.hash_pool + 32ull * (id - HASH_ID_BASE) : A.ref + 32ull * id;
}
__device__ __forceinline__ uint32_t ref_len_of(const ArenaView& A, uint32_t id) { return id >= HASH_ID_BASE ? 32u : (uint32_t)A.ref_len[id]; }

// ------------------------------------------------------------------ keccak batch -------------
// Message i = data[offsets[i * stride] .. offsets[i * stride + 1]): stride 1 for a packed batch
// (n + 1 offsets), stride 2 for explicit (begin, end) pairs.  Unit = 128 bytes of the message.

template <int B>
__global__ void __launch_bounds__(B) keccak256_batch_kernel(const uint8_t* __restrict__ data, const uint64_t* __restrict__ offsets,
                                                            uint32_t stride, uint32_t n, uint8_t* __restrict__ out) {
  __shared__ uint32_t smem[PPD_STAGE_WORDS * B];
  const uint32_t i = blockIdx.x * B + threadIdx.x;
  bool busy = i < n;
  Stage<B> s;
  s.init(smem);
  uint64_t a[25];
#pragma unroll
  for (int k = 0; k < 25; k++) a[k] = 0;
  const uint8_t* p = data;
  uint64_t left = 0;
  if (busy) {
    const uint64_t m_begin = offsets[(uint64_t)i * stride], m_end = offsets[(uint64_t)i * stride + 1];
    p = data + m_begin;
    left = m_end - m_begin;
  }
  for (;;) {
    bool last = false;
    if (busy) {
      while (s.bytes() < 136 && left) {
        uint32_t take = left < 128 ? (uint32_t)left : 128u;
        emit_bytes(s, p, take);
        p += take;
        left -= take;
      }
      last = s.bytes() < 136;
      if (last) s.pad();
      absorb_stage<B>(a, s);
    }
    if (!__any_sync(FULL, busy)) break;
    keccak_f1600(a);
    if (busy) {
      if (last) {
        uint4 x, y;
        digest_words(a, x, y);
        uint4* o = reinterpret_cast<uint4*>(out + 32ull * i);
        o[0] = x, o[1] = y;
        busy = false;
      } else {
        s.consume_block();
      }
    }
  }
}

// ------------------------------------------------------------------ trie level hashing -------
// One thread per node of the level (ids through `order`, which the host sorts by level and, inside
// a level, by node class so that the lanes of a warp run the same number of permutations).
//
// Unit list per kind (every unit <= 133 bytes, so the 272-byte stage never overflows):
//   LEAF          0: list header, hex-prefix key, value header   1..: 128 bytes of the value
//   LEAF_ACCOUNT  0: list header, hex-prefix key, string + list headers, nonce
//                 1: balance, storage root, code hash
//   EXT           0: list header, hex-prefix key, child ref
//   BRANCH        0: list header   1..: three children each with the empty slots before them (the last
//                 unit also carries the trailing empty slots and the empty value)
//   ROOT          0: the child's raw RLP (only when it is shorter than 32 bytes) or 0x80
//
// Gathers: a LEAF's value units and a BRANCH's child units go through the thread's gather slot.  Before
// the permutation of a block, the thread starts cp.async copies of the unit the next fill begins with
// (a leaf's next <= 128 value bytes, a branch's next three child refs), so the loads overlap the
// permutation instead of following it.  A unit the fill needs beyond that one is gathered and waited
// for on the spot.  A branch's child ids sit in the slot from the prologue on (chunks 6-9), so a unit
// needs no reload of child_pool.  The other kinds put all their units into the first block.
static constexpr int GATHER_CHUNKS = 10;  // branch: 3 refs (chunks 0-5) + 16 child ids (6-9); leaf: <= 144 bytes (0-8)
static constexpr uint32_t GATHER_IDS = 6;

template <int B>
using HashGather = Gather<B, GATHER_CHUNKS>;
template <int B>
constexpr uint32_t hash_smem_bytes() {
  return 4u * PPD_STAGE_WORDS * B + HashGather<B>::BYTES;
}

extern __shared__ uint4 hash_smem[];  // the block's stages, then its gather slots

template <int B>
__global__ void __launch_bounds__(B, 4) hash_level_kernel(ArenaView A, const uint32_t* __restrict__ order, uint32_t begin, uint32_t end) {
  uint32_t* smem = reinterpret_cast<uint32_t*>(hash_smem);
  const uint32_t slot = begin + blockIdx.x * B + threadIdx.x;
  uint32_t hashed = 0, perms = 0, enc_bytes = 0;
  bool busy = false, force_hash = false;
  // Persistent per-node state is kept small (the 50 state registers dominate): pointers are
  // re-derived from the record where they are used.
  uint32_t id = 0;
  uint4 rec = make_uint4(NK_HASH, 0, 0, 0);
  uint32_t payload = 0, nunit = 0, total = 0, unit = 0;
  // LEAF: vlen, vhdr   LEAF_ACCOUNT: vlen, nn | nb << 8 | apayload << 16   BRANCH: slots left, walk state
  uint32_t v0 = 0, v1 = 0;
  uint32_t gathered = 0;  // the unit whose source bytes are in the gather slot (0: none)
  HashGather<B> G;
  G.init(smem + PPD_STAGE_WORDS * B);
#define KIND (rec.x & 0xff)
#define NIB_START ((rec.x >> 8) & 0xff)
#define NIB_LEN ((rec.x >> 16) & 0xff)
#define MY_REF (A.ref + 32ull * id)

  if (slot < end) {
    id = order ? __ldg(order + slot) : slot;
    rec = __ldg(reinterpret_cast<const uint4*>(A.nodes) + id);
    const uint8_t* copy_src = nullptr;
    busy = true;
    switch (KIND) {
      case NK_LEAF: {
        const uint8_t* val = A.val_pool + rec.z;
        v0 = rec.w;
        v1 = (v0 == 1 && __ldg(val) < 0x80) ? 0 : len_prefix_size(v0);
        payload = hex_prefix_str_size(NIB_LEN) + v1 + v0;
        nunit = 1 + ((v0 + 127) >> 7);
        break;
      }
      case NK_LEAF_ACCOUNT: {
        const AccountRec* acc = A.accounts + rec.z;
        uint32_t nn = u256_sig_bytes(acc->nonce);
        uint32_t nb = u256_sig_bytes(acc->balance);
        uint32_t apayload = u256_str_size(acc->nonce, nn) + u256_str_size(acc->balance, nb) + 66;  // >= 68
        v0 = len_prefix_size(apayload) + apayload;                                                 // rlp(AccountRlp) >= 70
        v1 = nn | (nb << 8) | (apayload << 16);
        payload = hex_prefix_str_size(NIB_LEN) + len_prefix_size(v0) + v0;
        nunit = 2;
        break;
      }
      case NK_EXT: {
        uint32_t clen = ref_len_of(A, rec.z);
        payload = hex_prefix_str_size(NIB_LEN) + (clen == 32 ? 33 : clen);
        nunit = 1;
        break;
      }
      case NK_BRANCH: {
        const uint32_t* ch = A.child_pool + rec.y;
        const uint32_t mask = rec.z & 0xffff;
        const uint32_t k = __popc(mask);
        // all child ids, then all lengths: two batches of independent loads
        uint32_t cid[16];
#pragma unroll
        for (int j = 0; j < 16; j++) cid[j] = (uint32_t)j < k ? __ldg(ch + j) : NODE_EMPTY;
        payload = 17 - k;  // empty slots and the empty value
        uint32_t hashed_kids = 0;  // bit j: compact child j is referenced by hash
#pragma unroll
        for (int j = 0; j < 16; j++) {
          uint32_t cl = cid[j] == NODE_EMPTY ? 0u : ref_len_of(A, cid[j]);
          payload += cl == 32 ? 33u : cl;
          hashed_kids |= (cl == 32 ? 1u : 0u) << j;
        }
#pragma unroll
        for (int q = 0; q < 4; q++) sts128(G.chunk(GATHER_IDS + q), make_uint4(cid[4 * q], cid[4 * q + 1], cid[4 * q + 2], cid[4 * q + 3]));
        v0 = mask;               // slots still to emit
        v1 = hashed_kids << 16;  // | compact index of the next child << 8 | next slot
        nunit = 1 + (k + 2) / 3;
        break;
      }
      case NK_ROOT: {
        force_hash = true;
        if (rec.z != NODE_EMPTY && ref_len_of(A, rec.z) == 32) copy_src = ref_ptr(A, rec.z);
        nunit = 1;
        break;
      }
      default:
        busy = false;
        break;
    }
    if (copy_src) {
      const uint4* src = reinterpret_cast<const uint4*>(copy_src);
      uint4 x = __ldcg(src), y = __ldcg(src + 1);
      uint4* o = reinterpret_cast<uint4*>(MY_REF);
      o[0] = x;
      o[1] = y;
      A.ref_len[id] = 32;
      busy = false;
    }
    total = KIND == NK_ROOT ? 0 : len_prefix_size(payload) + payload;
  }
  const bool inline_ref = !force_hash && total < 32;

  // starts the copies of unit u >= 1 of a LEAF or a BRANCH into the gather slot (v0, v1: the walk state before u)
  auto gather = [&](uint32_t u) {
    if (KIND == NK_LEAF) {
      const uint32_t off = (u - 1) << 7;
      const uintptr_t p = reinterpret_cast<uintptr_t>(A.val_pool + rec.z + off);
      const uint8_t* q = reinterpret_cast<const uint8_t*>(p & ~(uintptr_t)15);  // (16-byte granules that hold a value byte)
      const uint32_t n_chunks = ((uint32_t)(p & 15) + min(128u, v0 - off) + 15) >> 4;
      for (uint32_t c = 0; c < n_chunks; c++) cp_async16(G.chunk(c), q + 16 * c);
    } else {
      const uint32_t j0 = (v1 >> 8) & 0xff, n_kids = min(3u, (uint32_t)__popc(v0));
      for (uint32_t t = 0; t < n_kids; t++) {
        const uint8_t* r = ref_ptr(A, G.word(4 * GATHER_IDS + j0 + t));
        cp_async16(G.chunk(2 * t), r);
        cp_async16(G.chunk(2 * t + 1), r + 16);
      }
    }
    cp_async_commit();
  };

  Stage<B> s;
  s.init(smem);
  uint64_t a[25];
#pragma unroll
  for (int k = 0; k < 25; k++) a[k] = 0;

  for (;;) {
    bool permute = false, last = false;
    if (busy) {
      // ---- fill: append whole units until a rate block is complete ----
      while (s.bytes() < 136 && unit < nunit) {
        if (unit > 0 && (KIND == NK_LEAF || KIND == NK_BRANCH) && gathered != unit) {
          gather(unit);
          cp_async_wait_all();
        }
        gathered = 0;
        switch (KIND) {
          case NK_LEAF:
            if (unit == 0) {
              emit_len_prefix(s, payload, 0xc0, 0xf7);
              emit_hex_prefix_str(s, A.key_pool + rec.y, NIB_START, NIB_LEN, 1);
              if (v1) emit_len_prefix(s, v0, 0x80, 0xb7);
            } else {
              const uint32_t off = (unit - 1) << 7;
              const uint32_t in_chunk = (uint32_t)(reinterpret_cast<uintptr_t>(A.val_pool + rec.z + off) & 15);
              const uint32_t w0 = in_chunk >> 2;
              emit_words(s, [&](uint32_t i) { return G.word(w0 + i); }, in_chunk & 3, min(128u, v0 - off));
            }
            break;
          case NK_LEAF_ACCOUNT: {
            const AccountRec* acc = A.accounts + rec.z;
            if (unit == 0) {
              emit_len_prefix(s, payload, 0xc0, 0xf7);
              emit_hex_prefix_str(s, A.key_pool + rec.y, NIB_START, NIB_LEN, 1);
              emit_len_prefix(s, v0, 0x80, 0xb7);
              emit_len_prefix(s, v1 >> 16, 0xc0, 0xf7);
              emit_u256_str(s, acc->nonce, v1 & 0xff);
            } else {
              emit_u256_str(s, acc->balance, (v1 >> 8) & 0xff);
              uint32_t src = acc->storage_src;
              emit_ref_at(s, src == NODE_EMPTY ? acc->storage_root : A.ref + 32ull * src, 32);
              emit_ref_at(s, acc->code_hash, 32);
            }
            break;
          }
          case NK_EXT:
            emit_len_prefix(s, payload, 0xc0, 0xf7);
            emit_hex_prefix_str(s, A.key_pool + rec.y, NIB_START, NIB_LEN, 0);
            emit_ref_at(s, ref_ptr(A, rec.z), ref_len_of(A, rec.z));
            break;
          case NK_BRANCH:
            if (unit == 0) {
              emit_len_prefix(s, payload, 0xc0, 0xf7);
            } else {
              // three children per unit, walked in compact order so that the lanes of a warp emit
              // their j-th child together whatever slots the children sit in
              uint32_t j0 = (v1 >> 8) & 0xff, next_slot = v1 & 0xff;
#pragma unroll
              for (int t = 0; t < 3; t++) {
                const uint32_t nib = v0 ? (uint32_t)__ffs(v0) - 1 : 16u;
                v0 &= v0 - 1;
                if (nib < 16) {
                  emit_empty_run(s, nib - next_slot);
                  const uint32_t len = ((v1 >> (16 + j0 + t)) & 1) ? 32u : ref_len_of(A, G.word(4 * GATHER_IDS + j0 + t));
                  emit_ref(s, lds128(G.chunk(2 * t)), lds128(G.chunk(2 * t + 1)), len);
                  next_slot = nib + 1;
                }
              }
              if (v0 == 0) emit_empty_run(s, 17 - next_slot);  // trailing empty slots and the empty value
              v1 = (v1 & 0xffff0000u) | ((j0 + 3) << 8) | next_slot;
            }
            break;
          default:  // NK_ROOT over Node::Empty or over a node whose encoding is < 32 bytes
            if (rec.z == NODE_EMPTY)
              s.put_byte(0x80);
            else
              emit_ref_at(s, ref_ptr(A, rec.z), ref_len_of(A, rec.z));
            break;
        }
        unit++;
      }
      if (inline_ref) {
        // the whole encoding (< 32 bytes) sits at the front of the stage: it is the ref
        uint4 x, y;
        inline_ref_words(s, total, x, y);
        uint4* o = reinterpret_cast<uint4*>(MY_REF);
        o[0] = x, o[1] = y;
        A.ref_len[id] = (uint8_t)total;
        busy = false;
      } else {
        last = s.bytes() < 136;
        if (last) s.pad();
        absorb_stage<B>(a, s);
        permute = true;
        // the next fill starts with unit `unit`: its loads run under the permutation
        if (!last && unit < nunit && (KIND == NK_LEAF || KIND == NK_BRANCH)) {
          gather(unit);
          gathered = unit;
        }
      }
    }
    if (!__any_sync(FULL, permute)) break;
    keccak_f1600(a);  // the single permutation site: the whole warp, converged
    cp_async_wait_all();
    if (permute) {
      perms++;
      if (last) {
        uint4 x, y;
        digest_words(a, x, y);
        uint4* o = reinterpret_cast<uint4*>(MY_REF);
        o[0] = x, o[1] = y;
        A.ref_len[id] = 32;
        hashed = 1;
        enc_bytes = KIND == NK_ROOT ? (rec.z == NODE_EMPTY ? 1u : ref_len_of(A, rec.z)) : total;
        busy = false;
      } else {
        s.consume_block();
      }
    }
  }
  add_counters(A.counters, hashed, perms, enc_bytes);
#undef KIND
#undef NIB_START
#undef NIB_LEN
#undef MY_REF
}

// ------------------------------------------------------------------ launchers ----------------

static constexpr int KB = 128;

void launch_keccak256_batch(const uint8_t* data, const uint64_t* offsets, uint32_t n, uint8_t* out, cudaStream_t st) {
  if (!n) return;
  keccak256_batch_kernel<KB><<<(n + KB - 1) / KB, KB, 0, st>>>(data, offsets, 1, n, out);
}
void launch_keccak256_ranges(const uint8_t* data, const uint64_t* begin_end, uint32_t n, uint8_t* out, cudaStream_t st) {
  if (!n) return;
  keccak256_batch_kernel<KB><<<(n + KB - 1) / KB, KB, 0, st>>>(data, begin_end, 2, n, out);
}
// ------------------------------------------------------------------ counting sort by a small key ----
// order[] = ids counting-sorted by a key of at most 4096 values: arena nodes by (level, class), so that inside a
// level nodes of one kind and one permutation count are adjacent, and the builder's branches by (depth, children);
// either way the lanes of a warp do the same work.  Three launches: per-CTA shared-memory histograms flushed to
// bins[], an exclusive scan of the bins, and a scatter in which every CTA reserves one range per key it holds.  The
// order inside a bucket is whatever the atomics give (hashing does not care).
static constexpr int OS_THREADS = 256, OS_PER = 8;  // items per CTA = 2048

__device__ __forceinline__ uint32_t node_class(const NodeRec& r) {
  const uint32_t kind = r.w0 & 0xff;
  if (kind == NK_BRANCH) return 40 + ((__popc(r.a1 & 0xffff) - 1) & 15);  // by child count
  if (kind == NK_ROOT) return 56;
  uint32_t perms = 1;
  if (kind == NK_LEAF) {
    const uint32_t nl = (r.w0 >> 16) & 0xff;
    perms = ((nl < 2 ? 1 : 2 + (nl >> 1)) + r.a2 + 6) / 136 + 1;  // header bytes over-estimated by at most 3
  }
  return kind * 8 + (perms > 8 ? 7 : perms - 1);
}

// A sort key: Key::of(a, b, j) = the bucket of item j, read from the arrays a and b (kernel parameters, so that they
// keep __restrict__ and are read through the read-only path).

// (level, class) of arena node j
struct LevelClassKey {
  static __device__ __forceinline__ uint32_t of(const NodeRec* __restrict__ nodes, const uint16_t* __restrict__ level, uint32_t j) {
    return (uint32_t)level[j] * 64u + node_class(nodes[j]);
  }
};

// (depth, number of children) of builder branch b: deepest depth first, then child counts ascending.  Lanes of a warp
// then walk the same number of children and run the same number of permutations (a branch with k hashed children
// encodes to 33 k + (16 - k) + 1 payload bytes: 1 rate block up to k = 3, 2 up to 7, 3 up to 12, else 4).
struct BranchKey {
  static __device__ __forceinline__ uint32_t of(const uint8_t* __restrict__ depth, const uint32_t* __restrict__ nchild_minus_1, uint32_t b) {
    return (63u - depth[b]) * 16 + min(nchild_minus_1[b], 15u);
  }
};

// after an update: the branches it hashes as BranchKey has them, then those whose refs it copied, one bucket per depth
struct UpdateBranchKey {
  static __device__ __forceinline__ uint32_t of(const uint8_t* __restrict__ depth, const uint32_t* __restrict__ nchild, uint32_t b) {
    const uint32_t c = nchild[b];
    return (c & BRANCH_CLEAN) ? BRANCH_BINS + 63u - depth[b] : (63u - depth[b]) * 16 + min(c, 15u);
  }
};

// The items sorted are first .. first + n (n read from *n_dev - first when n_dev is given: the txn loop's node count is
// only known on the device); keys[] and order[] are indexed from 0, order[] holds item ids.
template <class Key, class A, class B>
__global__ void __launch_bounds__(OS_THREADS) order_hist_kernel(const A* __restrict__ a, const B* __restrict__ b, uint32_t n, uint32_t n_bins,
                                                                uint16_t* __restrict__ keys, uint32_t* __restrict__ bins, uint32_t first,
                                                                const uint32_t* __restrict__ n_dev) {
  extern __shared__ uint32_t sh[];
  if (n_dev) n = min(n, *n_dev - first);
  if (blockIdx.x * (OS_THREADS * OS_PER) >= n) return;
  for (uint32_t k = threadIdx.x; k < n_bins; k += OS_THREADS) sh[k] = 0;
  __syncthreads();
  const uint32_t base = blockIdx.x * (OS_THREADS * OS_PER);
#pragma unroll
  for (int q = 0; q < OS_PER; q++) {
    const uint32_t i = base + q * OS_THREADS + threadIdx.x;
    if (i < n) {
      const uint32_t key = min(Key::of(a, b, first + i), n_bins - 1);
      keys[i] = (uint16_t)key;
      atomicAdd(&sh[key], 1u);
    }
  }
  __syncthreads();
  for (uint32_t k = threadIdx.x; k < n_bins; k += OS_THREADS)
    if (sh[k]) atomicAdd(&bins[k], sh[k]);
}

__global__ void __launch_bounds__(OS_THREADS) order_scatter_kernel(const uint16_t* __restrict__ keys, uint32_t n, uint32_t n_bins,
                                                                   uint32_t* __restrict__ cursor, uint32_t* __restrict__ order, uint32_t first,
                                                                   const uint32_t* __restrict__ n_dev) {
  extern __shared__ uint32_t sh[];  // [n_bins] counts, then this CTA's base per key
  if (n_dev) n = min(n, *n_dev - first);
  if (blockIdx.x * (OS_THREADS * OS_PER) >= n) return;
  for (uint32_t k = threadIdx.x; k < n_bins; k += OS_THREADS) sh[k] = 0;
  __syncthreads();
  const uint32_t base = blockIdx.x * (OS_THREADS * OS_PER);
  uint32_t key[OS_PER], rank[OS_PER];
#pragma unroll
  for (int q = 0; q < OS_PER; q++) {
    const uint32_t i = base + q * OS_THREADS + threadIdx.x;
    key[q] = i < n ? keys[i] : 0xffffffffu;
    rank[q] = i < n ? atomicAdd(&sh[key[q]], 1u) : 0u;
  }
  __syncthreads();
  for (uint32_t k = threadIdx.x; k < n_bins; k += OS_THREADS)
    if (sh[k]) sh[k] = atomicAdd(&cursor[k], sh[k]);
  __syncthreads();
#pragma unroll
  for (int q = 0; q < OS_PER; q++) {
    const uint32_t i = base + q * OS_THREADS + threadIdx.x;
    if (i < n) order[sh[key[q]] + rank[q]] = first + i;
  }
}

// ---- copies by kernel (see CopyBatch) ----
__global__ void copy_segments_kernel(CopyBatch B) {
  const uint32_t s = blockIdx.y;
  uint8_t* d = reinterpret_cast<uint8_t*>(B.dst[s]);
  const uint8_t* p = reinterpret_cast<const uint8_t*>(B.src[s]);
  const unsigned long long n = B.bytes[s];
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x, nt = (unsigned long long)gridDim.x * blockDim.x;
  const uintptr_t both = reinterpret_cast<uintptr_t>(d) | reinterpret_cast<uintptr_t>(p);
  unsigned long long done = 0;
  if ((both & 15) == 0) {
    const unsigned long long nv = n / 16;
    for (unsigned long long i = tid; i < nv; i += nt) reinterpret_cast<uint4*>(d)[i] = reinterpret_cast<const uint4*>(p)[i];
    done = nv * 16;
  } else if ((both & 3) == 0) {
    const unsigned long long nv = n / 4;
    for (unsigned long long i = tid; i < nv; i += nt) reinterpret_cast<uint32_t*>(d)[i] = reinterpret_cast<const uint32_t*>(p)[i];
    done = nv * 4;
  }
  for (unsigned long long i = done + tid; i < n; i += nt) d[i] = p[i];
}
void launch_copy_segments(const CopyBatch& B, cudaStream_t st) {
  if (!B.n) return;
  unsigned long long most = 0;
  for (uint32_t k = 0; k < B.n; k++) most = B.bytes[k] > most ? B.bytes[k] : most;
  uint32_t gx = (uint32_t)((most + 16 * 256 * 4 - 1) / (16 * 256 * 4));
  gx = gx < 1 ? 1 : (gx > 32 ? 32 : gx);
  copy_segments_kernel<<<dim3(gx, B.n), 256, 0, st>>>(B);
}
__global__ void store_u32x2_kernel(uint32_t* dst, uint32_t a, uint32_t b) { dst[0] = a, dst[1] = b; }
void launch_store_u32x2(uint32_t* dst, uint32_t a, uint32_t b, cudaStream_t st) { store_u32x2_kernel<<<1, 1, 0, st>>>(dst, a, b); }

// bins: [n_bins] zeroed by the caller; on return bins[k] = end of bucket k (the scatter advances the cursors)
template <class Key, class A, class B>
void counting_sort(const A* a, const B* b, uint32_t n, uint32_t n_bins, uint16_t* keys, uint32_t* bins, uint32_t* order, cudaStream_t st,
                   uint32_t first, const uint32_t* n_dev) {
  if (!n) return;
  const uint32_t blocks = (n + OS_THREADS * OS_PER - 1) / (OS_THREADS * OS_PER);
  order_hist_kernel<Key><<<blocks, OS_THREADS, 4 * n_bins, st>>>(a, b, n, n_bins, keys, bins, first, n_dev);
  exclusive_scan_small(bins, n_bins, st);
  order_scatter_kernel<<<blocks, OS_THREADS, 4 * n_bins, st>>>(keys, n, n_bins, bins, order, first, n_dev);
}
void launch_order_by_level_class(const NodeRec* nodes, const uint16_t* level, uint32_t n, uint32_t n_bins, uint16_t* keys, uint32_t* bins,
                                 uint32_t* order, cudaStream_t st, uint32_t first, const uint32_t* n_dev) {
  counting_sort<LevelClassKey>(nodes, level, n, n_bins, keys, bins, order, st, first, n_dev);
}
void launch_order_branches(const uint8_t* depth, const uint32_t* nchild_minus_1, uint32_t nb, uint16_t* keys, uint32_t* bins, uint32_t* order,
                           cudaStream_t st) {
  counting_sort<BranchKey>(depth, nchild_minus_1, nb, BRANCH_BINS, keys, bins, order, st, 0, nullptr);
}
void launch_order_update_branches(const uint8_t* depth, const uint32_t* nchild, uint32_t nb, uint16_t* keys, uint32_t* bins, uint32_t* order,
                                  cudaStream_t st) {
  counting_sort<UpdateBranchKey>(depth, nchild, nb, UPDATE_BRANCH_BINS, keys, bins, order, st, 0, nullptr);
}

// Stage and gather slots exceed the 48 KB of static shared memory: the kernel takes them as dynamic shared memory,
// with the carveout at its maximum so that four 128-thread CTAs (4 x (54 + 1) KB of the SM's 228 KB) share an SM.
static bool hash_level_ready() {
  static const bool once = [] {
    bool ok = cudaFuncSetAttribute(hash_level_kernel<KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hash_smem_bytes<KB>()) == cudaSuccess;
    ok &= cudaFuncSetAttribute(hash_level_kernel<KB>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared) == cudaSuccess;
    return ok;
  }();
  return once;
}

void launch_hash_level(const ArenaView& A, const uint32_t* order, uint32_t begin, uint32_t end, cudaStream_t st) {
  if (end <= begin) return;
  hash_level_ready();
  uint32_t n = end - begin;
  hash_level_kernel<KB><<<(n + KB - 1) / KB, KB, hash_smem_bytes<KB>(), st>>>(A, order, begin, end);
}

}  // namespace ppd
