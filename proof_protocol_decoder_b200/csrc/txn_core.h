// txn_core.h — the txn loop of decoding.rs:80-177 on the node arena, written once for the device and for a CPU
// check harness (tests/cpp/txn_core_check.cpp emulates the thread block phase by phase; the product only ever
// runs the __device__ instantiation, ppd_txn.cu).
//
// What it replaces (SURVEY.md rows a11-a13, a19): per txn
//   create_minimal_partial_tries_needed_by_txn  decoding.rs:179-217, 551-602  -> every key's walk marks what it visits (batch_walk)
//   apply_deltas_to_trie_state                  decoding.rs:219-292, 431-456  -> two batched trie updates (Batch)
//   eth_trie_utils insert / delete / get        (SURVEY.md A.2)               -> path copies on the arena in HBM
//
// Design.  The shape of a trie never depends on a hash, so every version of every trie of a block is built
// before anything is hashed, as new records appended to the arena (nodes are immutable, old versions stay
// addressable, unchanged subtrees are shared).  One thread block runs the whole txn loop of one block; the txns
// are sequential, the keys of one txn are parallel:
//   * every key the txn accesses or writes walks the version before the txn ONCE: the walk marks the nodes it visits
//     (the subset of the txn keeps those expanded) and records the nodes it passes (its path) and where it ends (its
//     terminal: an empty slot, a leaf, a hashed-out node, or the middle of an extension);
//   * keys are sorted per trie (op_rank) with the LCP of neighbours (op_lcp), so "the keys that pass through
//     the node at depth d on my path" is a contiguous range and its first key, the OWNER, is the one whose LCP
//     with its predecessor is < d;
//   * terminals are resolved by their owners (a new leaf, an overwrite, a split, a removal);
//   * path nodes are re-assembled bottom-up, one barrier per depth: the owner of a branch gathers the results
//     of the children its range touched, creates the new version once (not once per key), and collapses a
//     branch left with one child exactly as delete does (SURVEY.md A.2).
// The result of a batch is the trie the reference reaches by applying the same writes one by one (a Merkle
// Patricia trie is canonical for its items, hashed-out subtrees counting as items), without the versions in
// between, which nobody observes (the reference hashes a trie once per txn, decoding.rs:458-464).
// Anything the reference would report as an error (an insert through a hashed-out node, a subset key running
// into one, a key that is a prefix of another ...) raises a flag; the block is then redone by the host path
// (host_txn.cu), which reports errors in the reference's order.
#pragma once
#include <cstdint>

#include "../../include/ppd_flat.h"
#include "arena.h"

// Everything is force-inlined on the device: the View (a struct of ~60 pointers and sizes) must never be an object in
// memory that some store through a uint32_t* might alias, or every use of a field becomes a reload behind every store
// (measured: the sixteen child-table stores of one node took sixteen dependent round trips).
#if defined(__CUDACC__)
#define PPD_HD __host__ __device__ __forceinline__
#define PPD_INLINE
#else
#define PPD_HD
#define PPD_INLINE inline
#endif

namespace ppd {
namespace txn {

static const uint32_t T_UNCHANGED = 0xfffffffeu;  // batch result: the subtree did not change
static const uint32_t ST_ABSENT = 0xfffffffeu;    // AcctState::storage: no entry in the storage map (decoding.rs:572-582)
static const uint32_t NONE = 0xfffffffdu;
static const uint32_t HASH_BASE = 0x80000000u, HASH_END = 0xf0000000u;
static const uint32_t MARK_SLOTS_T = 16;  // == MARK_SLOTS (ppd_kernels.h): touched slots per key
static const uint32_t PATH_CAP = 15;      // nodes a key may pass before its terminal (the path and the terminal fill the key's touched slots)
static const uint32_t OWNER_TXN_TRIE = 0xffffff01u, OWNER_RECEIPT_TRIE = 0xffffff02u, OWNER_STATE_TRIE = 0xffffff03u;
static const uint32_t TRF_STATE_WRITE = 0x100u;   // TxnTrace::flags: the trace changes the account (processed_block_trace.rs:238-256)
static const uint32_t TRF_MIN_KEYS = 0x200u;      // a written slot key has a leading zero byte: decoding.rs:235 hashes the shortened key

enum : uint32_t {
  TXF_OK = 0,
  TXF_INSERT_INTO_HASH = 1,  // PPD_PANIC_INSERT_INTO_HASH_NODE in the reference
  TXF_KEY_PREFIX = 2,        // PPD_PANIC_KEY_IS_PREFIX_OF_KEY
  TXF_MARK_INTO_HASH = 3,    // PPD_ERR_MISSING_KEYS_CREATING_SUB_PARTIAL_TRIE
  TXF_MARK_SLOTS = 4,        // a marking walk longer than its slots
  TXF_PATH_DEPTH = 5,        // a batched key passes more than PATH_CAP nodes
  TXF_NODES_FULL = 6,
  TXF_CHILDREN_FULL = 7,
  TXF_KEYS_FULL = 8,
  TXF_NOT_ACCOUNT = 9,       // PPD_ERR_ACCOUNT_DECODE
  TXF_DUP_KEY = 10,          // the same key twice in one batch (only a malformed FlatBlock has that)
  TXF_SHORT_HADDR = 11,      // PPD_PANIC_H256_FROM_SLICE
  TXF_LEVELS = 12,
  TXF_WITHDRAWAL = 13,       // PPD_ERR_MISSING_WITHDRAWAL_ACCOUNT / account decode
  TXF_STACK = 14,
  TXF_SHARED_TRIE = 15,
  TXF_PATH_TABLE = 16,       // the path-node table of a txn is full      // the by-root join gives two accounts the SAME witnessed trie: the host path clones it, as the reference does
};

enum : uint8_t { OP_DEL = 0, OP_PUT_LEAF = 1, OP_PUT_ACCOUNT = 2, OP_NONE = 3 };  // OP_NONE: a key that is only accessed
enum : uint8_t { SOP_MARK = 1 };  // SOp::pad: the key is one the txn ACCESSES (its walk is a marking walk of create_trie_subset)
enum : uint8_t { TK_EMPTY = 0, TK_LEAF_SAME = 1, TK_LEAF_OTHER = 2, TK_HASH = 3, TK_DIVERGE = 4, TK_BAD = 5 };

// One key of a txn, in sorted order within its trie: an accessed key (marking walk only), a write (which is an access
// too, unless decoding.rs:235 hashed a shortened slot key for it), a delete.
struct SOp {
  uint32_t koff;   // key in key_pool
  uint32_t a1, a2; // PUT_LEAF: value offset, length; PUT_ACCOUNT: account record
  uint32_t owner;  // trace whose storage trie it writes, or OWNER_*
  uint8_t klen;    // nibbles
  int8_t lcp;      // common prefix (nibbles) with the previous op of the same trie; -1 for the first
  uint8_t kind;
  uint8_t pad;
};

// One TxnTrace (trace_protocol.rs:152-183) as the host lays it out for the device.  Offsets are into the FlatBlock.
struct TxnTrace {
  uint32_t flags, txn;
  uint32_t off_addr, off_balance, off_nonce;
  uint32_t off_reads, n_reads, off_writes, n_writes;
  uint32_t code_off, code_len;
  uint32_t m_reads, m_wfull, m_wmin, m_code;  // digest indices (the address digest of trace t is digest t)
  uint32_t op0;    // first round-1 key of the trace: its slot reads, its slot writes (twice with TRF_MIN_KEYS: the full and the shortened key)
  uint32_t n_keys; // how many
  uint32_t rec;    // account record its state write fills
  uint32_t val0;   // val_pool offset of its first written value (36 bytes apart)
  uint32_t acct;   // (device) account table slot
  uint32_t rank;   // (device) position among the txn's traces sorted by hashed address
  uint32_t pad;
};

struct TxnDesc {
  uint32_t trace_begin, trace_end;
  uint32_t touched_base;  // first slot of the IR's touched list
  uint32_t seg_tries;     // plan segments: +0 state, +1 transactions, +2 receipts sub-trie
  uint32_t seg_storage;   // +2r: hashed address of the r-th account in sorted order, +2r+1: its storage sub-trie
  uint32_t seg_roots;     // +0 state, +1 transactions, +2 receipts root after the txn
  uint32_t key_off, key_nibs;  // Nibbles::from_bytes_be(rlp(txn_idx)), decoding.rs:190
  uint32_t off_txn_bytes, len_txn_bytes, off_receipt, len_receipt;  // FlatBlock offsets
  uint32_t val_txn, val_receipt;                                    // val_pool offsets
  uint32_t op1_begin, op1_end;  // round 1: storage writes of every trace, then the txn / receipt inserts
  uint32_t op2_begin, op2_end;  // round 2: state writes and self-destructs
};

struct AcctState {
  uint32_t storage;    // root of the account's storage trie in PartialTrieState, NODE_EMPTY, or ST_ABSENT
  uint32_t root_node;  // NK_ROOT node over `storage`, or NONE
  uint32_t pre_rec;    // the account's record in the pre-image, or NONE
  uint32_t owner;      // (table) first trace that claimed the slot, or 0xffffffff
};

enum { XR_INITIAL_STATE = 0, XR_EMPTY = 1, XR_FINAL_STATE = 2, XR_FINAL_TXN = 3, XR_FINAL_RECEIPT = 4, XR_AFTER_WITHDRAWALS = 5 };
struct Cursors {
  uint32_t n_nodes, n_children, key_bytes;  // allocation cursors
  uint32_t flag, flag_txn;                  // first TXF_* raised and where
  uint32_t state_root, txn_root, receipt_root;
  uint32_t max_level;
  uint32_t roots[6];  // NK_ROOT nodes the dummy entries refer to (XR_*), created when the loop ends
  uint32_t state_before_withdrawals;
  uint32_t pc_count;  // path-node table entries handed out (when the table is in HBM)
  uint32_t pad0;
  // SM clocks per phase of the loop, summed over txns: setup, walks, announce, storage / txn / receipt tries back up,
  // account records, state trie back up, root nodes
  unsigned long long phase_clocks[8];
};

// One withdrawal (decoding.rs:404-428): balance += amount on the account of the hashed address
struct Withdrawal {
  uint32_t m_addr;      // digest index of the address
  uint32_t off_amount;  // FlatBlock offset of the 32-byte amount
  uint32_t rec;         // account record the updated account fills
  uint32_t pad;
};

// A node on the path of some key of the running txn.
struct PathNode {
  uint32_t kids[16];  // a branch's children as they are before the txn, overwritten by the children that changed; an extension: [0] = its child's result
  uint32_t node;      // the arena node
  uint32_t lv;        // level the new version needs: the old node's, raised by changed children
  uint32_t pending;   // children (groups of keys) that have not reported yet: the last one to report re-assembles the node
  uint32_t owner;     // first key through the node (index into the batch)
  uint32_t changed;
  uint32_t pad[3];
};

// Everything the loop touches.  All pointers are device pointers (host pointers in the CPU harness).
// The part of a view the loop kernel re-points: the cursors and the scratch of the running txn live in shared memory while
// it runs (ppd_txn.cu); everything else of the view is read-only kernel-parameter space.  SCR(v) is how the loop reads it.
struct Scratch {
  // allocation cursors: &cur->n_nodes ..., or shared-memory copies of them while the loop kernel runs (an allocation is
  // then a shared-memory atomic instead of a round trip to L2)
  uint32_t *a_nodes, *a_children, *a_keys, *a_max_level;
  // scratch of the running txn, indexed by key (round-1 keys first, then the state keys); in shared memory when the
  // txn's keys fit (ppd_txn.cu), else in HBM
  uint32_t* path_node;  // [keys][PATH_CAP] nodes passed, root first
  uint32_t* path_pc;    // [keys][PATH_CAP] the node's entry in the path-node table below, for the levels the key leads
  uint8_t* path_depth;  // [keys][PATH_CAP] nibble depth at which the node starts | 0x80 for an extension
  uint8_t* plen;        // [keys]
  uint32_t* tnode;      // [keys] terminal node
  uint32_t* tpc;        // [keys] its path-node entry when the key leaves an extension half way
  uint8_t* tdepth;      // [keys]
  uint8_t* tkind;       // [keys]
  uint32_t* key_hi;     // [keys] nibbles 0..7 of the key, most significant first (child slots without a key load)
  SOp* sh_ops;          // [keys] copy of the txn's keys when the scratch is in shared memory, else nullptr
  // the path-node table of the running txn: one entry per distinct node some key passes (or leaves half way), made by
  // the node's OWNER (the first key through it) during the walk; children report to it on their way up.  The first
  // pc_fast entries live in shared memory, the rest in HBM.
  PathNode* pc_fast;
  PathNode* pc_slow;
  uint32_t pc_n_fast, pc_n_slow;
  uint32_t* pc_count;   // entries handed out (reset per txn)
  uint32_t* pc_map;     // [pc_map_mask + 1] node id -> entry + 1 (open addressing; 0 = free), reset per txn
  uint32_t* pc_map_key;
  uint32_t pc_map_mask;
};

struct View {
  // arena (mutable: the loop appends)
  NodeRec* nodes;
  uint16_t* level;
  uint8_t* key_pool;
  uint8_t* val_pool;
  const uint8_t* hash_pool;
  uint32_t* child_pool;
  AccountRec* accounts;
  uint32_t cap_nodes, cap_children, cap_keys;
  // inputs
  const uint8_t* flat;
  TxnTrace* traces;
  const TxnDesc* txns;
  uint32_t n_txns, n_traces;
  uint32_t dig_base;         // key_pool offset of digest 0 (32 bytes each)
  uint32_t rec_base, val_base;  // TxnTrace::rec / val0 and Withdrawal::rec count from here (accounts[], val_pool)
  AcctState* acct;           // account table
  uint32_t* pre_slot;        // per pre-image account: its slot of the account table once a trace touched it (else >= NONE)
  const Withdrawal* withdrawals;
  uint32_t n_withdrawals;
  const uint8_t* pre_flags;  // per pre-image account: bit0 storage root != EMPTY_TRIE_HASH
  SOp* ops1;
  SOp* ops2;
  // plan (outputs)
  uint32_t* touched;
  uint32_t* seg_a;
  uint32_t* seg_b;
  Scratch s;  // what the loop kernel re-points to shared memory (SCR below)
  Cursors* cur;
  // PPD_LOOP_PROF builds: per-thread event log of one txn (clock, thread << 16 | event)
  unsigned long long* evlog;
  uint32_t* evcount;
  uint32_t ev_txn, ev_cap;
};

#if defined(__CUDA_ARCH__)
// (the loop kernel keeps its Scratch at the start of its dynamic shared memory)
__device__ __forceinline__ Scratch& scratch_of(const View&) {
  extern __shared__ __align__(16) uint8_t ppd_loop_smem[];
  return *reinterpret_cast<Scratch*>(ppd_loop_smem);
}
#define SCR(v) ppd::txn::scratch_of(v)
#else
#define SCR(v) ((v).s)
#endif

// the by-root join of accounts to witnessed storage tries (compact_to_partial_trie.rs:167-190), ppd_txn.cu
// one block's loop as the kernel takes it (ppd_txn.cu: txn_loop_kernel; an array of these per launch)
struct LoopTask {
  View v;
  uint32_t initial_state, use_shared, pad[2];
};

struct JoinView {
  const uint32_t* acct_list;  // [n_acct][5] as ParseEmit writes it: leaf, storage trie root, its NK_ROOT node, flags, code index
  uint32_t n_acct;
  const uint8_t* ref;         // refs of the pre-image nodes (the storage roots are hashed before the loop)
  uint32_t* slot_owner;       // [table_mask + 1], 0xffffffff = free
  uint32_t* slot_best;        // [table_mask + 1], 1 + the last account that witnesses a trie with this root
  uint32_t table_mask;
  uint32_t* join_storage;     // [n_acct] out
  uint32_t* join_root;        // [n_acct] out
  uint8_t* pre_flags;         // [n_acct] out
  uint32_t* flag;             // &Cursors::flag
  // the by-address join of a direct pre-image (FlatBlock kind 2) instead, when keep is set: the hashed addresses of its
  // storage map; slot_owner then holds map indices, slot_best[0] 1 + the last account whose witnessed trie is empty
  const uint8_t* keep;        // [n_keep][32], or null
  uint32_t n_keep;
};

PPD_HD PPD_INLINE bool is_hash_id(uint32_t n) { return n >= HASH_BASE && n < HASH_END; }

// ---- the execution context: how threads of the block see shared counters ------------------------------------
// Device: a thread block.  Harness: one "thread" at a time.
struct Ctx {
  const View& v;
  uint32_t tid, nthreads;
  long long* sh_clock;  // shared: clock at the last phase boundary
};

#if defined(__CUDA_ARCH__) && defined(PPD_LOOP_PROF)
#define PPD_EV(v, txn, tid, id)                                                        \
  do {                                                                                 \
    if ((v).evlog && (txn) == (v).ev_txn) {                                            \
      const uint32_t ev_i = atomicAdd((v).evcount, 1u);                                \
      if (ev_i < (v).ev_cap) (v).evlog[2 * ev_i] = clock64(), (v).evlog[2 * ev_i + 1] = ((unsigned long long)(tid) << 16) | (id); \
    }                                                                                  \
  } while (0)
#else
#define PPD_EV(v, txn, tid, id) ((void)0)
#endif
#if defined(__CUDA_ARCH__)
#define PPD_PREFETCH(p) asm volatile("prefetch.global.L1 [%0];" ::"l"(p))
#define PPD_FENCE_BLOCK() __threadfence_block()
#define PPD_ATOMIC_SUB(p, x) atomicSub((p), (x))
#define PPD_ATOMIC_ADD(p, x) atomicAdd((p), (x))
#define PPD_ATOMIC_MAX(p, x) atomicMax((p), (x))
#define PPD_ATOMIC_CAS(p, c, x) atomicCAS((p), (c), (x))
#else
PPD_HD PPD_INLINE uint32_t host_atomic_add(uint32_t* p, uint32_t x) {
  uint32_t o = *p;
  *p = o + x;
  return o;
}
PPD_HD PPD_INLINE uint32_t host_atomic_max(uint32_t* p, uint32_t x) {
  uint32_t o = *p;
  if (x > o) *p = x;
  return o;
}
PPD_HD PPD_INLINE uint32_t host_atomic_cas(uint32_t* p, uint32_t c, uint32_t x) {
  uint32_t o = *p;
  if (o == c) *p = x;
  return o;
}
#define PPD_FENCE_BLOCK() ((void)0)
#define PPD_PREFETCH(p) ((void)0)
#define PPD_ATOMIC_SUB(p, x) ppd::txn::host_atomic_add((p), 0u - (x))
#define PPD_ATOMIC_ADD(p, x) ppd::txn::host_atomic_add((p), (x))
#define PPD_ATOMIC_MAX(p, x) ppd::txn::host_atomic_max((p), (x))
#define PPD_ATOMIC_CAS(p, c, x) ppd::txn::host_atomic_cas((p), (c), (x))
#endif

PPD_HD PPD_INLINE void raise(const View& v, uint32_t why, uint32_t txn) {
  if (PPD_ATOMIC_CAS(&v.cur->flag, 0u, why) == 0u) v.cur->flag_txn = txn;
}

// ---- arena primitives (the device form of host_arena.h) -------------------------------------------------------
PPD_HD PPD_INLINE uint32_t key_nib(const View& v, uint32_t koff, uint32_t i) {
  const uint32_t b = v.key_pool[koff + (i >> 1)];
  return (i & 1) ? (b & 15u) : (b >> 4);
}
PPD_HD PPD_INLINE uint32_t lvl(const View& v, uint32_t n) { return (n == NODE_EMPTY || n >= HASH_BASE) ? 0u : (uint32_t)v.level[n]; }
PPD_HD PPD_INLINE uint32_t kind_of(const View& v, uint32_t n) { return is_hash_id(n) ? (uint32_t)NK_HASH : (v.nodes[n].w0 & 0xffu); }
PPD_HD PPD_INLINE uint32_t w0(uint32_t kind, uint32_t start, uint32_t len) { return kind | (start << 8) | (len << 16); }

PPD_HD PPD_INLINE uint32_t push_node(const View& v, const NodeRec& r, uint32_t lv) {
  uint32_t id = PPD_ATOMIC_ADD(SCR(v).a_nodes, 1u);
  if (id >= v.cap_nodes) {
    raise(v, TXF_NODES_FULL, 0);
    id = v.cap_nodes - 1;  // a sink slot: the block is redone anyway
  }
  if (lv > 0xfff0u) raise(v, TXF_LEVELS, 0), lv = 0xfff0u;
  v.nodes[id] = r;
  v.level[id] = (uint16_t)lv;
  PPD_ATOMIC_MAX(SCR(v).a_max_level, lv);
  return id;
}
PPD_HD PPD_INLINE uint32_t alloc_children(const View& v, uint32_t k) {
  uint32_t at = PPD_ATOMIC_ADD(SCR(v).a_children, k);
  if (at + k > v.cap_children) {
    raise(v, TXF_CHILDREN_FULL, 0);
    at = v.cap_children - 16;
  }
  return at;
}
// up to 32 bytes of the key pool from byte offset `off`, as 8 words in memory order (byte j of the string: word j / 4,
// bits 8 * (j % 4)): aligned word loads, all in flight together, shifted into place.  Words past the first `nbytes` bytes
// are zero.
PPD_HD PPD_INLINE void load_key_words(const View& v, uint32_t off, uint32_t nbytes, uint32_t* w) {
  const uint32_t* base = reinterpret_cast<const uint32_t*>(v.key_pool) + (off >> 2);
  const uint32_t sh = 8u * (off & 3u), nw = (nbytes + (off & 3u) + 3u) >> 2;
  uint32_t a[9];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (uint32_t j = 0; j < 9; j++) a[j] = j < nw ? base[j] : 0u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (uint32_t j = 0; j < 8; j++) w[j] = sh ? (a[j] >> sh) | (a[j + 1] << (32u - sh)) : a[j];
}
PPD_HD PPD_INLINE uint32_t ctz32(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return (uint32_t)__ffs((int)x) - 1u;
#else
  return (uint32_t)__builtin_ctz(x);
#endif
}
// the number of leading nibbles (at most m) that key a from nibble sa and key b from nibble sb have in common
PPD_HD PPD_INLINE uint32_t common_prefix(const View& v, uint32_t ka, uint32_t sa, uint32_t kb, uint32_t sb, uint32_t m) {
  if (m == 0) return 0;
  if (((sa ^ sb) & 1u) == 0 && m <= 64u - (sa & 1u)) {
    // same parity (always, for nodes on a key's own path): both strings loaded whole, one round trip, compared in registers
    const uint32_t odd = sa & 1u, nb = (odd + m + 1u) >> 1;
    uint32_t wa[8], wb[8];
    load_key_words(v, ka + (sa >> 1), nb, wa);
    load_key_words(v, kb + (sb >> 1), nb, wb);
    uint32_t cp = 2u * nb;  // (in nibbles from the first byte; no difference found: everything loaded is equal)
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 7; j >= 0; j--) {
      uint32_t x = wa[j] ^ wb[j];
      if (j == 0 && odd) x &= ~0xf0u;  // the first byte's high nibble is before the start
      if (x) {
        const uint32_t byte = ctz32(x) >> 3, bx = (x >> (8u * byte)) & 0xffu;
        cp = 2u * (4u * (uint32_t)j + byte) + ((bx & 0xf0u) ? 0u : 1u);
      }
    }
    cp -= odd;
    return cp < m ? cp : m;
  }
  uint32_t i = 0;
  while (i < m && key_nib(v, ka, sa + i) == key_nib(v, kb, sb + i)) i++;
  return i;
}
// nibble i of a key held in registers (load_key_words from the key's first byte)
PPD_HD PPD_INLINE uint32_t nib_of_words(const uint32_t* w, uint32_t i) {
  const uint32_t j = i >> 3;
  uint32_t x = w[0];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (uint32_t z = 1; z < 8; z++)
    if (j == z) x = w[z];
  const uint32_t byte = (x >> (8u * ((i >> 1) & 3u))) & 0xffu;
  return (i & 1u) ? (byte & 15u) : (byte >> 4);
}
PPD_HD PPD_INLINE uint32_t child_at(const View& v, const NodeRec& br, uint32_t nib) {
  const uint32_t mask = br.a1 & 0xffffu, bit = 1u << nib;
  if (!(mask & bit)) return NODE_EMPTY;
#if defined(__CUDA_ARCH__)
  return v.child_pool[br.a0 + __popc(mask & (bit - 1))];
#else
  return v.child_pool[br.a0 + __builtin_popcount(mask & (bit - 1))];
#endif
}
PPD_HD PPD_INLINE uint32_t popc16(uint32_t m) {
#if defined(__CUDA_ARCH__)
  return __popc(m & 0xffffu);
#else
  return (uint32_t)__builtin_popcount(m & 0xffffu);
#endif
}

// A node id with its level.  The level of a new node is 1 + the largest level of what it reads; the creators carry the
// levels of what they have just made instead of reading them back (a read back is a trip to L2, and sixteen of them in
// a row, one per child of a new branch, were most of the re-assembly's time).
struct NL {
  uint32_t id, lv;
};
PPD_HD PPD_INLINE NL new_leaf_for(const View& v, const SOp& o, uint32_t start) {
  const uint32_t len = o.klen - start;
  if (o.kind == OP_PUT_ACCOUNT) {
    const uint32_t src = v.accounts[o.a1].storage_src;
    const uint32_t lv = src == NODE_EMPTY ? 0u : lvl(v, src) + 1u;
    return NL{push_node(v, NodeRec{w0(NK_LEAF_ACCOUNT, start, len), o.koff, o.a1, 0}, lv), lv};
  }
  return NL{push_node(v, NodeRec{w0(NK_LEAF, start, len), o.koff, o.a1, o.a2}, 0), 0};
}
PPD_HD PPD_INLINE NL new_ext(const View& v, uint32_t koff, uint32_t start, uint32_t len, NL child) {
  return NL{push_node(v, NodeRec{w0(NK_EXT, start, len), koff, child.id, 0}, child.lv + 1u), child.lv + 1u};
}
PPD_HD PPD_INLINE uint32_t new_root(const View& v, uint32_t child) {
  return push_node(v, NodeRec{w0(NK_ROOT, 0, 0), 0, child, 0}, child == NODE_EMPTY ? 0u : lvl(v, child) + 1u);
}
// the same leaf payload under a different key range
PPD_HD PPD_INLINE NL releaf(const View& v, uint32_t leaf, uint32_t leaf_lv, uint32_t koff, uint32_t start, uint32_t len) {
  NodeRec r = v.nodes[leaf];
  r.w0 = w0(r.w0 & 0xffu, start, len);
  r.a0 = koff;
  return NL{push_node(v, r, leaf_lv), leaf_lv};
}
// branch of level lv from 16 slots (NODE_EMPTY = none); at least two are set
PPD_HD PPD_INLINE NL new_branch16(const View& v, const uint32_t* kids, uint32_t lv) {
  uint32_t mask = 0, k = 0;
  for (uint32_t i = 0; i < 16; i++)
    if (kids[i] != NODE_EMPTY) mask |= 1u << i, k++;
  const uint32_t base = alloc_children(v, k);
  for (uint32_t i = 0, j = 0; i < 16; i++)
    if (kids[i] != NODE_EMPTY) v.child_pool[base + j++] = kids[i];
  return NL{push_node(v, NodeRec{w0(NK_BRANCH, 0, 0), base, mask, 0}, lv), lv};
}
// copy of branch `br` with slot `nib` set to `child` (never NODE_EMPTY here)
PPD_HD PPD_INLINE NL branch_with(const View& v, uint32_t br, uint32_t nib, NL child) {
  const NodeRec r = v.nodes[br];
  uint32_t lv = v.level[br];
  const uint32_t mask = r.a1 & 0xffffu, bit = 1u << nib;
  const uint32_t k = popc16(mask), rk = popc16(mask & (bit - 1)), has = (mask & bit) ? 1u : 0u;
  const uint32_t nk = k - has + 1u, base = alloc_children(v, nk);
  uint32_t old[16];
  for (uint32_t i = 0; i < 16; i++) old[i] = i < k ? v.child_pool[r.a0 + i] : 0u;  // (all in flight together)
  for (uint32_t i = 0; i < rk; i++) v.child_pool[base + i] = old[i];
  v.child_pool[base + rk] = child.id;
  for (uint32_t i = rk + has; i < k; i++) v.child_pool[base + i - has + 1u] = old[i];
  if (child.lv + 1u > lv) lv = child.lv + 1u;
  return NL{push_node(v, NodeRec{w0(NK_BRANCH, 0, 0), base, mask | bit, 0}, lv), lv};
}
// an extension (ek, es, el) over `child`, merged into the child when that is a leaf / an extension (delete's collapse)
PPD_HD PPD_INLINE NL collapse_ext(const View& v, uint32_t ek, uint32_t es, uint32_t el, NL child) {
  const uint32_t k = kind_of(v, child.id);
  if (k == NK_EXT) {
    const NodeRec c = v.nodes[child.id];  // (the merged extension reads what the child read: the child's level)
    return NL{push_node(v, NodeRec{w0(NK_EXT, ((c.w0 >> 8) & 0xffu) - el, ((c.w0 >> 16) & 0xffu) + el), c.a0, c.a1, 0}, child.lv), child.lv};
  }
  if (k == NK_LEAF || k == NK_LEAF_ACCOUNT) {
    const NodeRec c = v.nodes[child.id];
    return releaf(v, child.id, child.lv, c.a0, ((c.w0 >> 8) & 0xffu) - el, ((c.w0 >> 16) & 0xffu) + el);
  }
  return new_ext(v, ek, es, el, child);
}
// the single child left in slot `nib` of a branch at depth `pos` on the path of key `koff`
PPD_HD PPD_INLINE NL collapse_branch(const View& v, uint32_t koff, uint32_t pos, uint32_t nib, NL other) {
  const uint32_t k = kind_of(v, other.id);
  if (k == NK_EXT || k == NK_LEAF || k == NK_LEAF_ACCOUNT) return collapse_ext(v, 0, pos, 1, other);  // their own keys spell the nibble
  // a key that runs through the surviving child: the path's first `pos` nibbles, then its slot
  const uint32_t nb = pos / 2 + 2;
  uint32_t pk = PPD_ATOMIC_ADD(SCR(v).a_keys, nb);
  if (pk + nb > v.cap_keys) {
    raise(v, TXF_KEYS_FULL, 0);
    pk = v.cap_keys - 40;
  }
  for (uint32_t i = 0; i <= pos / 2; i++) v.key_pool[pk + i] = v.key_pool[koff + i];
  uint8_t* last = v.key_pool + pk + pos / 2;
  *last = (pos & 1) ? (uint8_t)((*last & 0xf0u) | nib) : (uint8_t)(nib << 4);
  v.key_pool[pk + pos / 2 + 1] = 0;
  return new_ext(v, pk, pos, 1, other);
}

// ---- insert of one key below `base`, which sits at depth `depth` on the key's path (HostArena::insert, iterative) ----
PPD_HD PPD_INLINE NL split_at(const View& v, const SOp& o, uint32_t pos, uint32_t cp, uint32_t existing_nib, NL existing, uint32_t txn) {
  const uint32_t at = pos + cp;
  if (at >= o.klen) {
    raise(v, TXF_KEY_PREFIX, txn);
    return existing;
  }
  const uint32_t new_nib = key_nib(v, o.koff, at);
  uint32_t kids[16];
  for (int i = 0; i < 16; i++) kids[i] = NODE_EMPTY;
  const NL leaf = new_leaf_for(v, o, at + 1);
  kids[existing_nib] = existing.id;
  kids[new_nib] = leaf.id;
  const NL br = new_branch16(v, kids, (existing.lv > leaf.lv ? existing.lv : leaf.lv) + 1u);
  return cp == 0 ? br : new_ext(v, o.koff, pos, cp, br);
}
PPD_HD PPD_INLINE NL insert_one(const View& v, NL base, uint32_t depth, const SOp& o, uint32_t txn) {
  uint32_t st_node[PATH_CAP + 1];
  uint8_t st_nib[PATH_CAP + 1];  // 0..15: branch slot; 0xff: extension
  uint32_t sp = 0, node = base.id, pos = depth;
  NL result = base;
  for (;;) {
    if (node == NODE_EMPTY) {
      result = new_leaf_for(v, o, pos);
      break;
    }
    const uint32_t k = kind_of(v, node);
    if (k == NK_HASH || k == NK_ROOT) {
      raise(v, TXF_INSERT_INTO_HASH, txn);
      return base;
    }
    const NodeRec r = v.nodes[node];
    const uint32_t ns = (r.w0 >> 8) & 0xffu, nl = (r.w0 >> 16) & 0xffu;
    if (k == NK_BRANCH) {
      if (pos >= o.klen || sp == PATH_CAP + 1) {
        raise(v, pos >= o.klen ? TXF_KEY_PREFIX : TXF_STACK, txn);
        return base;
      }
      const uint32_t nib = key_nib(v, o.koff, pos);
      st_node[sp] = node, st_nib[sp] = (uint8_t)nib, sp++;
      node = child_at(v, r, nib);
      pos++;
    } else if (k == NK_EXT) {
      const uint32_t avail = o.klen - pos, m = avail < nl ? avail : nl;
      const uint32_t cp = common_prefix(v, r.a0, ns, o.koff, pos, m);
      if (cp == nl) {
        if (sp == PATH_CAP + 1) {
          raise(v, TXF_STACK, txn);
          return base;
        }
        st_node[sp] = node, st_nib[sp] = 0xff, sp++;
        node = r.a1;
        pos += nl;
      } else {
        const uint32_t rem = nl - cp - 1;
        const NL child{r.a1, lvl(v, r.a1)};
        const NL existing = rem == 0 ? child : new_ext(v, r.a0, ns + cp + 1, rem, child);
        result = split_at(v, o, pos, cp, key_nib(v, r.a0, ns + cp), existing, txn);
        break;
      }
    } else {  // leaves
      const uint32_t avail = o.klen - pos, m = avail < nl ? avail : nl;
      const uint32_t cp = common_prefix(v, r.a0, ns, o.koff, pos, m);
      if (cp == nl && nl == avail) {
        result = new_leaf_for(v, o, pos);  // overwrite
      } else if (cp == nl) {
        raise(v, TXF_KEY_PREFIX, txn);
        return base;
      } else {
        const NL existing = releaf(v, node, node == base.id ? base.lv : (uint32_t)v.level[node], r.a0, ns + cp + 1, nl - cp - 1);
        result = split_at(v, o, pos, cp, key_nib(v, r.a0, ns + cp), existing, txn);
      }
      break;
    }
  }
  while (sp) {
    sp--;
    if (st_nib[sp] == 0xff) {
      const NodeRec r = v.nodes[st_node[sp]];
      result = new_ext(v, r.a0, (r.w0 >> 8) & 0xffu, (r.w0 >> 16) & 0xffu, result);
    } else {
      result = branch_with(v, st_node[sp], st_nib[sp], result);
    }
  }
  return result;
}

// ---- one batched update: ops[0 .. n) sorted by (trie, key); scratch entries base .. base + n ----------------------
struct Batch {
  const SOp* ops;
  uint32_t n;
  uint32_t base;  // index of ops[0] in the scratch arrays
  uint32_t txn;
};

// The nodes on the path of key i at depth <= shared_depth(b, i) are on the path of a neighbouring key as well (keys are
// sorted: a node at depth d is shared with the predecessor / successor exactly when the LCP with it is >= d); the nodes
// below are this key's alone.  -1: the key is alone in its trie.
PPD_HD PPD_INLINE int shared_depth(const Batch& b, uint32_t i) {
  const int prev = (int)b.ops[i].lcp, next = i + 1 < b.n ? (int)b.ops[i + 1].lcp : -1;
  return prev > next ? prev : next;
}
PPD_HD PPD_INLINE uint32_t trie_root_of(const View& v, uint32_t owner) {
  if (owner == OWNER_STATE_TRIE) return v.cur->state_root;
  if (owner == OWNER_TXN_TRIE) return v.cur->txn_root;
  if (owner == OWNER_RECEIPT_TRIE) return v.cur->receipt_root;
  return v.acct[v.traces[owner].acct].storage;
}

PPD_HD PPD_INLINE PathNode& pc_at(const View& v, uint32_t idx) { return idx < SCR(v).pc_n_fast ? SCR(v).pc_fast[idx] : SCR(v).pc_slow[idx - SCR(v).pc_n_fast]; }
PPD_HD PPD_INLINE uint32_t pc_hash(uint32_t node) { return node * 2654435761u; }
// the owner of a path node makes its table entry during the walk and publishes it under the node id; the node's child
// table and level are loaded afterwards, all entries in parallel (pc_fill)
PPD_HD PPD_INLINE uint32_t pc_make(const View& v, uint32_t node, const NodeRec& r, bool is_branch, uint32_t owner, uint32_t txn) {
  uint32_t idx = PPD_ATOMIC_ADD(SCR(v).pc_count, 1u);
  if (idx >= SCR(v).pc_n_fast + SCR(v).pc_n_slow) {
    raise(v, TXF_PATH_TABLE, txn);
    return NONE;
  }
  PathNode& p = pc_at(v, idx);
  p.kids[0] = r.a0, p.kids[1] = is_branch ? (r.a1 & 0xffffu) : 0x10000u;  // (until pc_fill replaces them)
  p.node = node, p.lv = 0, p.pending = 0, p.owner = owner, p.changed = 0;
  uint32_t h = pc_hash(node) & SCR(v).pc_map_mask;
  for (;;) {
    const uint32_t prev = PPD_ATOMIC_CAS(&SCR(v).pc_map_key[h], 0xffffffffu, node);
    if (prev == 0xffffffffu || prev == node) break;  // (a node has one owner: `prev == node` does not happen)
    h = (h + 1) & SCR(v).pc_map_mask;
  }
  SCR(v).pc_map[h] = idx + 1u;
  return idx;
}
// per table entry: the node's children as they are before the txn (sixteen independent loads), and its level
PPD_HD PPD_INLINE void pc_fill(const View& v, uint32_t idx) {
  PathNode& p = pc_at(v, idx);
  const uint32_t a0 = p.kids[0], m = p.kids[1];
  const uint32_t old_lv = v.level[p.node];
  if (m & 0x10000u) {  // an extension: [0] will hold its child's result
    p.kids[0] = T_UNCHANGED, p.kids[1] = 0;
  } else {
    const uint32_t mask = m & 0xffffu;
    // sixteen independent loads (the slot of a child in the compact table follows from the mask alone)
    uint32_t x[16];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (uint32_t nib = 0; nib < 16; nib++) x[nib] = ((mask >> nib) & 1u) ? v.child_pool[a0 + popc16(mask & ((1u << nib) - 1u))] : NODE_EMPTY;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (uint32_t nib = 0; nib < 16; nib++) p.kids[nib] = x[nib];
  }
  p.lv = old_lv;
}
PPD_HD PPD_INLINE uint32_t pc_find(const View& v, uint32_t node) {
  uint32_t h = pc_hash(node) & SCR(v).pc_map_mask;
  for (;;) {
    const uint32_t k = SCR(v).pc_map_key[h];
    if (k == node) return SCR(v).pc_map[h] - 1u;
    if (k == 0xffffffffu) return NONE;
    h = (h + 1) & SCR(v).pc_map_mask;
  }
}

// The walk of key i down the current version of its trie.  It is the key's marking walk (the nodes it visits go to the
// IR's touched list: create_trie_subset keeps exactly those expanded) AND the first half of its write: the nodes passed
// and where the key ends are kept for the way back up.
PPD_HD PPD_INLINE void batch_walk(const Ctx& c, const Batch& b, uint32_t i, uint32_t* touched) {
  const View& v = c.v;
  PPD_EV(v, b.txn, c.tid, 1);
  const SOp o = b.ops[i];
  const uint32_t e = b.base + i;
  uint32_t node = trie_root_of(v, o.owner), pos = 0, pl = 0, nt = 0;
  uint32_t kw[8];  // the key, in registers: the nibble that picks a branch's child costs no load
  load_key_words(v, o.koff, (o.klen + 1u) >> 1, kw);
  uint32_t* pn = SCR(v).path_node + (size_t)e * PATH_CAP;
  uint8_t* pd = SCR(v).path_depth + (size_t)e * PATH_CAP;
  uint32_t tk = TK_EMPTY, tn = NODE_EMPTY, td = 0, tpc = NONE;
  const bool put = o.kind == OP_PUT_LEAF || o.kind == OP_PUT_ACCOUNT, mark = (o.pad & SOP_MARK) != 0;
  const int shared = shared_depth(b, i);
  for (;;) {
    if (node == NODE_EMPTY) {
      tk = TK_EMPTY, td = pos;
      break;
    }
    if (mark) touched[nt] = node;
    nt++;
    NodeRec r{NK_HASH, 0, 0, 0};
    if (!is_hash_id(node)) r = v.nodes[node];
    const uint32_t k = r.w0 & 0xffu;
    if (k == NK_HASH || k == NK_ROOT) {
      tk = TK_HASH, tn = node, td = pos;
      if (put) raise(v, TXF_INSERT_INTO_HASH, b.txn);
      if (mark && pos < o.klen) raise(v, TXF_MARK_INTO_HASH, b.txn);  // MissingKeysCreatingSubPartialTrie
      break;
    }
    const uint32_t ns = (r.w0 >> 8) & 0xffu, nl = (r.w0 >> 16) & 0xffu;
    const bool owner = (int)o.lcp < (int)pos && (int)pos <= shared;  // the first key through this node, when there are others
    if (k == NK_BRANCH) {
      if (pos >= o.klen || pl == PATH_CAP) {
        if (pos >= o.klen) {
          if (put) raise(v, TXF_KEY_PREFIX, b.txn);
        } else {
          raise(v, TXF_PATH_DEPTH, b.txn);
        }
        tk = TK_BAD, tn = node, td = pos;
        break;
      }
      pn[pl] = node, pd[pl] = (uint8_t)pos, pl++;
      if (owner) pc_make(v, node, r, true, i, b.txn);
      node = child_at(v, r, nib_of_words(kw, pos));
      pos++;
    } else if (k == NK_EXT) {
      const uint32_t avail = o.klen - pos, m = avail < nl ? avail : nl;
      const uint32_t cp = common_prefix(v, r.a0, ns, o.koff, pos, m);
      if (owner) tpc = pc_make(v, node, r, false, i, b.txn);
      if (cp == nl) {
        if (pl == PATH_CAP) {
          raise(v, TXF_PATH_DEPTH, b.txn);
          tk = TK_BAD, tn = node, td = pos;
          break;
        }
        pn[pl] = node, pd[pl] = (uint8_t)(pos | 0x80u), pl++;
        node = r.a1;
        pos += nl;
      } else {
        if (cp == avail && put) raise(v, TXF_KEY_PREFIX, b.txn);
        tk = TK_DIVERGE, tn = node, td = pos;
        break;
      }
    } else {
      const uint32_t avail = o.klen - pos, m = avail < nl ? avail : nl;
      const uint32_t cp = common_prefix(v, r.a0, ns, o.koff, pos, m);
      const bool same = cp == nl && nl == avail;
      if (!same && (cp == nl || cp == avail) && put) raise(v, TXF_KEY_PREFIX, b.txn);
      tk = same ? TK_LEAF_SAME : TK_LEAF_OTHER, tn = node, td = pos;
      break;
    }
  }
  if (nt > MARK_SLOTS_T) raise(v, TXF_MARK_SLOTS, b.txn);  // (unreachable: PATH_CAP + 1 slots)
  SCR(v).plen[e] = (uint8_t)pl;
  SCR(v).tnode[e] = tn, SCR(v).tdepth[e] = (uint8_t)td, SCR(v).tkind[e] = (uint8_t)tk;
  // the key's first eight nibbles, most significant first (short keys: zero nibbles after their end)
  SCR(v).key_hi[e] = (kw[0] << 24) | ((kw[0] & 0xff00u) << 8) | ((kw[0] >> 8) & 0xff00u) | (kw[0] >> 24);
  PPD_EV(v, b.txn, c.tid, 2);
}

// The canonical trie over a small group of sorted items that share their first `td` nibbles: the writes of one group
// (keys that end at the same place) plus, possibly, the leaf that was there.  One pass with a stack of open branches
// (no walk per item, no intermediate versions): what inserting the items one by one arrives at.  Returns false when the
// group is not of the plain kind (too many items, keys of different lengths): the caller then inserts one by one.
static const uint32_t GROUP_MAX = 12;
PPD_HD PPD_INLINE bool build_group(const View& v, const Batch& b, uint32_t first, uint32_t end, uint32_t td, uint32_t old_leaf, bool keep_old, NL* out, uint32_t txn) {
  // items: (key offset, op index or NONE for the old leaf), in key order, with the LCP (absolute) to the previous item
  uint32_t ik[GROUP_MAX + 1], iop[GROUP_MAX + 1];
  int il[GROUP_MAX + 2];
  uint32_t m = 0;
  NodeRec oldr{};
  uint32_t old_koff = 0, old_lv = 0;
  if (keep_old) {
    oldr = v.nodes[old_leaf];
    old_koff = oldr.a0;
    old_lv = v.level[old_leaf];
    if (((oldr.w0 >> 8) & 0xffu) + ((oldr.w0 >> 16) & 0xffu) != 64u) return false;
  }
  bool old_placed = !keep_old;
  int run_min = 127, prev_cpx = -1;
  for (uint32_t j = first; j < end; j++) {
    if (j > first && (int)b.ops[j].lcp < run_min) run_min = b.ops[j].lcp;
    const uint8_t kind = b.ops[j].kind;
    if (kind != OP_PUT_LEAF && kind != OP_PUT_ACCOUNT) continue;
    if (b.ops[j].klen != 64 || m + 2 > GROUP_MAX) return false;
    int l_prev = m == 0 ? (int)td - 1 : run_min;  // LCP with the previous write (the minimum over the keys skipped in between)
    if (!old_placed) {
      const int cpx = (int)td + (int)common_prefix(v, old_koff, td, b.ops[j].koff, td, 64 - td);
      if (cpx >= 64) return false;  // (an overwrite: the caller drops the old leaf)
      if (key_nib(v, old_koff, (uint32_t)cpx) < key_nib(v, b.ops[j].koff, (uint32_t)cpx)) {
        // the old leaf comes before this write
        ik[m] = old_koff, iop[m] = NONE, il[m] = m == 0 ? (int)td - 1 : prev_cpx, m++;
        old_placed = true;
        l_prev = cpx;
      } else {
        prev_cpx = cpx;
      }
    }
    ik[m] = b.ops[j].koff, iop[m] = j, il[m] = l_prev, m++;
    run_min = 127;
  }
  if (!old_placed) ik[m] = old_koff, iop[m] = NONE, il[m] = m == 0 ? (int)td - 1 : prev_cpx, m++;
  il[m] = (int)td - 1;
  if (m == 0) {
    *out = NL{NODE_EMPTY, 0};
    return true;
  }
  // stack of open branches
  uint32_t sd[GROUP_MAX + 1], slv[GROUP_MAX + 1], sk[GROUP_MAX + 1][16];
  uint32_t sp = 0;
  for (uint32_t k = 0; k < m; k++) {
    const int lc = il[k], ln = il[k + 1];
    const uint32_t s = (uint32_t)((lc > ln ? lc : ln) + 1);
    NL cur = iop[k] == NONE ? releaf(v, old_leaf, old_lv, old_koff, s, 64 - s) : new_leaf_for(v, b.ops[iop[k]], s);
    if (ln > lc) {  // a branch at depth ln opens with this leaf as its first child
      sd[sp] = (uint32_t)ln, slv[sp] = cur.lv + 1u;
      for (int z = 0; z < 16; z++) sk[sp][z] = NODE_EMPTY;
      sk[sp][key_nib(v, ik[k], (uint32_t)ln)] = cur.id;
      sp++;
      continue;
    }
    if (sp == 0) {  // a single item
      *out = cur;
      return true;
    }
    sk[sp - 1][key_nib(v, ik[k], (uint32_t)lc)] = cur.id;
    if (cur.lv + 1u > slv[sp - 1]) slv[sp - 1] = cur.lv + 1u;
    while (sp && (int)sd[sp - 1] > ln) {
      sp--;
      const uint32_t d = sd[sp];
      NL br = new_branch16(v, sk[sp], slv[sp]);
      const int parent = sp ? (int)sd[sp - 1] : (int)td - 1;
      const int p = parent > ln ? parent : ln;
      if (p < (int)d - 1) br = new_ext(v, ik[k], (uint32_t)(p + 1), d - (uint32_t)(p + 1), br);
      if (p < (int)td) {  // above the group: this is its top node
        *out = br;
        return true;
      }
      const uint32_t nib = key_nib(v, ik[k], (uint32_t)p);
      if (sp && p == parent) {
        sk[sp - 1][nib] = br.id;
        if (br.lv + 1u > slv[sp - 1]) slv[sp - 1] = br.lv + 1u;
      } else {
        sd[sp] = (uint32_t)p, slv[sp] = br.lv + 1u;
        for (int z = 0; z < 16; z++) sk[sp][z] = NODE_EMPTY;
        sk[sp][nib] = br.id;
        sp++;
        break;
      }
    }
  }
  raise(v, TXF_STACK, txn);  // (unreachable: the last item closes every open branch)
  return false;
}

// After every walk: a key looks up the table entry of every node on its path, and announces itself at the nodes whose
// child it LEADS (it is the first key of the group that goes into that child): every leader will report there, and the
// last report re-assembles the node.  A key leads the child of the branch at depth d when its LCP with its predecessor
// is <= d; the one child of an extension that ends at depth d' when it is < d'.  A key that leaves an extension half
// way announces itself there on its own account.
PPD_HD PPD_INLINE void batch_announce(const Ctx& c, const Batch& b, uint32_t i) {
  const View& v = c.v;
  const uint32_t e = b.base + i;
  const int lcp = (int)b.ops[i].lcp;
  const uint32_t pl = SCR(v).plen[e];
  const uint32_t* pn = SCR(v).path_node + (size_t)e * PATH_CAP;
  uint32_t* ppc = SCR(v).path_pc + (size_t)e * PATH_CAP;
  const uint8_t* pd = SCR(v).path_depth + (size_t)e * PATH_CAP;
  const int shared = shared_depth(b, i);
  bool leads = true;
  for (uint32_t t = pl; t-- > 0;) {
    const uint32_t d = pd[t] & 0x7fu;
    if ((int)d > shared) continue;  // this key's alone: no table entry (batch_climb rebuilds it in place)
    const uint32_t child_depth = (pd[t] & 0x80u) ? (t + 1 < pl ? (uint32_t)(pd[t + 1] & 0x7fu) : (uint32_t)SCR(v).tdepth[e]) : d + 1;
    const uint32_t idx = pc_find(v, pn[t]);
    ppc[t] = idx;
    leads = leads && lcp < (int)child_depth;  // (once the predecessor goes into the same child it does so at every node above)
    if (leads && idx != NONE) PPD_ATOMIC_ADD(&pc_at(v, idx).pending, 1u);
  }
  uint32_t tidx = NONE;
  if (SCR(v).tkind[e] == TK_DIVERGE && (int)SCR(v).tdepth[e] <= shared) {
    tidx = pc_find(v, SCR(v).tnode[e]);
    if (tidx != NONE) PPD_ATOMIC_ADD(&pc_at(v, tidx).pending, 1u);
  }
  SCR(v).tpc[e] = tidx;
}

// new version of the branch behind table entry p (the children that changed have been written into p.kids); koff / d: a
// key through the branch and the branch's depth
PPD_HD PPD_INLINE NL assemble_branch(const View& v, PathNode& p, uint32_t koff, uint32_t d) {
  uint32_t nk = 0, last = 0;
  for (uint32_t nib = 0; nib < 16; nib++)
    if (p.kids[nib] != NODE_EMPTY) nk++, last = nib;
  if (nk >= 2) return new_branch16(v, p.kids, p.lv);
  if (nk == 1) return collapse_branch(v, koff, d, last, NL{p.kids[last], lvl(v, p.kids[last])});  // (delete's collapse; rare)
  return NL{NODE_EMPTY, 0};
}
// new version of the extension behind table entry p (its child's result is in p.kids[0], with its level in [1]); the keys
// of its range that leave it half way split it
PPD_HD PPD_INLINE NL assemble_ext(const View& v, const Batch& b, PathNode& p, uint32_t d) {
  const NodeRec r = v.nodes[p.node];
  const uint32_t el = (r.w0 >> 16) & 0xffu;
  NL base{p.node, p.lv};
  bool changed = false;
  const uint32_t rj = p.kids[0];
  if (rj == NODE_EMPTY)
    base = NL{NODE_EMPTY, 0}, changed = true;
  else if (rj != T_UNCHANGED)
    base = collapse_ext(v, r.a0, d, el, NL{rj, p.kids[1]}), changed = true;
  for (uint32_t j = p.owner; j < b.n && (j == p.owner || (int)b.ops[j].lcp >= (int)d); j++)
    if (SCR(v).tkind[b.base + j] == TK_DIVERGE && SCR(v).tdepth[b.base + j] == d && (b.ops[j].kind == OP_PUT_LEAF || b.ops[j].kind == OP_PUT_ACCOUNT))
      base = insert_one(v, base, d, b.ops[j], b.txn), changed = true;
  return changed ? base : NL{T_UNCHANGED, 0};
}

PPD_HD PPD_INLINE void set_trie_root(const View& v, uint32_t owner, uint32_t r) {
  if (owner == OWNER_STATE_TRIE) {
    v.cur->state_root = r;
  } else if (owner == OWNER_TXN_TRIE) {
    v.cur->txn_root = r;
  } else if (owner == OWNER_RECEIPT_TRIE) {
    v.cur->receipt_root = r;
  } else {
    AcctState& a = v.acct[v.traces[owner].acct];
    a.storage = r, a.root_node = NONE;
  }
}

// ---- the part of a path that is one key's alone: rebuilt by that key's thread, node by node, without the table ----
// branch `node` at depth d with the child in slot `nib` replaced by the (changed) result `cur`; koff: a key through it
PPD_HD PPD_INLINE NL private_branch(const View& v, uint32_t node, uint32_t d, uint32_t nib, NL cur, uint32_t koff) {
  if (cur.id != NODE_EMPTY) return branch_with(v, node, nib, cur);
  const NodeRec r = v.nodes[node];
  const uint32_t lv = v.level[node];
  const uint32_t mask = r.a1 & 0xffffu, bit = 1u << nib;
  if (!(mask & bit)) return NL{T_UNCHANGED, 0};
  const uint32_t left = mask & ~bit, nk = popc16(left);
  if (nk >= 2) {  // the branch without the child
    const uint32_t base = alloc_children(v, nk), gone = popc16(mask & (bit - 1u));
    uint32_t old[16];
    for (uint32_t i = 0; i < 16; i++) old[i] = i <= nk ? v.child_pool[r.a0 + i] : 0u;  // (all in flight together)
    for (uint32_t i = 0; i < nk; i++) v.child_pool[base + i] = old[i < gone ? i : i + 1u];
    return NL{push_node(v, NodeRec{w0(NK_BRANCH, 0, 0), base, left, 0}, lv), lv};
  }
  if (nk == 1) {  // delete's collapse (SURVEY.md A.2)
    const uint32_t last = ctz32(left), kid = v.child_pool[r.a0 + popc16(mask & ((1u << last) - 1u))];
    return collapse_branch(v, koff, d, last, NL{kid, lvl(v, kid)});
  }
  return NL{NODE_EMPTY, 0};
}
// extension `node` at depth d over the (changed) result `cur` of its child
PPD_HD PPD_INLINE NL private_ext(const View& v, uint32_t node, uint32_t d, NL cur) {
  if (cur.id == NODE_EMPTY) return cur;
  const NodeRec r = v.nodes[node];
  return collapse_ext(v, r.a0, d, (r.w0 >> 16) & 0xffu, cur);
}

// The way back up of key i.  Its terminal is resolved by the first key of the group that ends there (a new leaf, an
// overwrite, a split, a removal).  That key reports the result to the node above; the LAST child to report to a node
// re-assembles it (a branch left with one child collapses as delete does, SURVEY.md A.2) and reports it to the node
// above in turn, on behalf of the node's whole range (every key of the range has the same nodes above).  No barrier
// and no scan of the range: a step is a handful of shared-memory operations plus the stores of the new node.  Whoever
// re-assembles the topmost node installs the trie's new root.
PPD_HD PPD_INLINE void batch_climb(const Ctx& c, const Batch& b, uint32_t i) {
  const View& v = c.v;
  const uint32_t e = b.base + i;
  const SOp& o = b.ops[i];
  const uint32_t tk = SCR(v).tkind[e], td = SCR(v).tdepth[e];
  const uint32_t* ppc = SCR(v).path_pc + (size_t)e * PATH_CAP;
  const uint8_t* pd = SCR(v).path_depth + (size_t)e * PATH_CAP;
  NL cur{T_UNCHANGED, 0};
  uint32_t t = SCR(v).plen[e];
  const int shared = shared_depth(b, i);
  if (tk == TK_DIVERGE && (int)td > shared) {
    // the only key at this extension, which it leaves half way: the split, in place
    if (o.kind == OP_PUT_LEAF || o.kind == OP_PUT_ACCOUNT) cur = insert_one(v, NL{SCR(v).tnode[e], (uint32_t)v.level[SCR(v).tnode[e]]}, td, o, b.txn);
  } else if (tk == TK_DIVERGE) {
    // one of the keys that leave the extension half way: it reports to the extension on its own account
    const uint32_t idx = SCR(v).tpc[e];
    if (idx == NONE) return;
    PathNode& p = pc_at(v, idx);
    PPD_FENCE_BLOCK();
    if (PPD_ATOMIC_SUB(&p.pending, 1u) != 1u) return;
    PPD_FENCE_BLOCK();
    cur = assemble_ext(v, b, p, td);
  } else {
    if ((int)o.lcp >= (int)td) return;  // shares the terminal with its predecessor: the group's first key reports
    if (tk == TK_EMPTY || tk == TK_LEAF_SAME || tk == TK_LEAF_OTHER) {
      bool any = false;  // nothing to do for a group of accessed-only keys (most groups): decided before anything is loaded
      for (uint32_t j = i; j < b.n && (j == i || (int)b.ops[j].lcp >= (int)td); j++) any |= b.ops[j].kind != OP_NONE;
      if (any) {
        NL base{NODE_EMPTY, 0};
        if (tk != TK_EMPTY) base = NL{SCR(v).tnode[e], (uint32_t)v.level[SCR(v).tnode[e]]};
        bool changed = false, keep_old = tk != TK_EMPTY;
        uint32_t end = i, n_put = 0;
        // the leaf that is there goes when its own key is deleted or overwritten; then the inserts (the order of distinct keys does not matter)
        for (uint32_t j = i; j < b.n && (j == i || (int)b.ops[j].lcp >= (int)td); j++, end++) {
          const uint8_t kind = b.ops[j].kind;
          if (kind == OP_DEL && SCR(v).tkind[b.base + j] == TK_LEAF_SAME) base = NL{NODE_EMPTY, 0}, changed = true, keep_old = false;
          if (kind == OP_PUT_LEAF || kind == OP_PUT_ACCOUNT) {
            n_put++, changed = true;
            if (SCR(v).tkind[b.base + j] == TK_LEAF_SAME) keep_old = false;
          }
        }
        NL built;
        if (n_put >= 2 && build_group(v, b, i, end, td, SCR(v).tnode[e], keep_old, &built, b.txn)) {
          base = built;
        } else {
          for (uint32_t j = i; j < end; j++)
            if (b.ops[j].kind == OP_PUT_LEAF || b.ops[j].kind == OP_PUT_ACCOUNT) base = insert_one(v, base, td, b.ops[j], b.txn);
        }
        if (changed) cur = base;
      }
    }
  }
  PPD_EV(v, b.txn, c.tid, 11);
  for (;;) {
    if (t == 0) {  // what this key carries is the new version of the whole trie
      if (cur.id != T_UNCHANGED) set_trie_root(v, o.owner, cur.id);
      return;
    }
    t--;
    const uint32_t d = pd[t] & 0x7fu;
    const bool is_ext = (pd[t] & 0x80u) != 0;
    if ((int)d > shared) {  // this key's alone
      if (cur.id != T_UNCHANGED) {
        const uint32_t node = SCR(v).path_node[(size_t)e * PATH_CAP + t];
        cur = is_ext ? private_ext(v, node, d, cur) : private_branch(v, node, d, d < 8 ? (SCR(v).key_hi[e] >> (28 - 4 * d)) & 15u : key_nib(v, o.koff, d), cur, o.koff);
      }
      continue;
    }
    const uint32_t idx = ppc[t];
    if (idx == NONE) return;  // (the table was full: a flag is up)
    PathNode& q = pc_at(v, idx);
    if (cur.id != T_UNCHANGED) {
      if (is_ext) {
        q.kids[0] = cur.id, q.kids[1] = cur.lv;
      } else {
        q.kids[d < 8 ? (SCR(v).key_hi[e] >> (28 - 4 * d)) & 15u : key_nib(v, o.koff, d)] = cur.id;
        if (cur.id != NODE_EMPTY) PPD_ATOMIC_MAX(&q.lv, cur.lv + 1u);
      }
      q.changed = 1;
    }
    PPD_FENCE_BLOCK();
    if (PPD_ATOMIC_SUB(&q.pending, 1u) != 1u) return;  // others have yet to report: the last of them carries on
    PPD_FENCE_BLOCK();
    PPD_EV(v, b.txn, c.tid, 12);
    if (is_ext)
      cur = assemble_ext(v, b, q, d);
    else if (q.changed)
      cur = assemble_branch(v, q, o.koff, d);
    else
      cur = NL{T_UNCHANGED, 0};
    PPD_EV(v, b.txn, c.tid, 13);
  }
}

// ---- op preparation (all txns at once, before the loop) -----------------------------------------------------
// 32-byte keys compare as big-endian numbers == bytewise
PPD_HD PPD_INLINE int cmp32(const uint8_t* a, const uint8_t* b) {
  for (int i = 0; i < 32; i++)
    if (a[i] != b[i]) return a[i] < b[i] ? -1 : 1;
  return 0;
}
PPD_HD PPD_INLINE int lcp_nibbles(const View& v, uint32_t ka, uint32_t na, uint32_t kb, uint32_t nb) {
  const uint32_t m = na < nb ? na : nb;
  uint32_t i = 0;
  while (i < m && key_nib(v, ka, i) == key_nib(v, kb, i)) i++;
  return (int)i;
}
PPD_HD PPD_INLINE const uint8_t* digest(const View& v, uint32_t m) { return v.key_pool + v.dig_base + 32ull * m; }

// per trace t: the byte ranges of the FlatBlock whose Keccak-256 the loop needs (utils.rs:11-13 call sites
// processed_block_trace.rs:219,234,277 and decoding.rs:235), as (begin, end) pairs indexed like the digests
PPD_HD PPD_INLINE void prep_msgs(const View& v, uint32_t t, uint64_t* se) {
  const TxnTrace& tr = v.traces[t];
  se[2 * t] = tr.off_addr, se[2 * t + 1] = tr.off_addr + 20ull;
  for (uint32_t k = 0; k < tr.n_reads; k++) se[2 * (tr.m_reads + k)] = tr.off_reads + 32ull * k, se[2 * (tr.m_reads + k) + 1] = tr.off_reads + 32ull * k + 32;
  for (uint32_t k = 0; k < tr.n_writes; k++) {
    const uint64_t key = tr.off_writes + 64ull * k;
    se[2 * (tr.m_wfull + k)] = key, se[2 * (tr.m_wfull + k) + 1] = key + 32;
    if (tr.flags & TRF_MIN_KEYS) {  // Nibbles::bytes_be() drops leading zero bytes (decoding.rs:235)
      uint32_t z = 0;
      while (z < 32 && v.flat[key + z] == 0) z++;
      se[2 * (tr.m_wmin + k)] = key + z, se[2 * (tr.m_wmin + k) + 1] = key + 32;
    }
  }
  if ((tr.flags & PPD_TR_CODE_WRITE) && !(tr.flags & PPD_TR_CODE_READ)) se[2 * tr.m_code] = tr.code_off, se[2 * tr.m_code + 1] = (uint64_t)tr.code_off + tr.code_len;
}

PPD_HD PPD_INLINE void prep_withdrawal_msg(const View& v, uint32_t w, uint64_t* se) {  // the address precedes the amount
  const Withdrawal wd = v.withdrawals[w];
  se[2 * wd.m_addr] = wd.off_amount - 20ull, se[2 * wd.m_addr + 1] = wd.off_amount;
}

// per trace t: its rank among the traces of its txn by hashed address, which is the place of its state key (and of its
// storage trie in the IR): every trace accesses its account (processed_block_trace.rs:267), some write it
PPD_HD PPD_INLINE void prep_trace(const View& v, uint32_t t) {
  TxnTrace& tr = v.traces[t];
  const TxnDesc& tx = v.txns[tr.txn];
  const uint8_t* me = digest(v, t);
  uint32_t rank = 0;
  for (uint32_t u = tx.trace_begin; u < tx.trace_end; u++) {
    if (u == t) continue;
    const int c = cmp32(digest(v, u), me);
    if (c == 0) raise(v, TXF_DUP_KEY, tr.txn);  // (TxnInfo.traces is a map: only a malformed FlatBlock repeats an address)
    if (c < 0 || (c == 0 && u < t)) rank++;
  }
  tr.rank = rank;
  if (me[0] == 0) raise(v, TXF_SHORT_HADDR, tr.txn);  // H256::from_slice(&nibbles.bytes_be()), decoding.rs:202
  SOp o;
  o.koff = v.dig_base + 32u * t, o.klen = 64, o.lcp = -1, o.pad = SOP_MARK;
  o.kind = (tr.flags & PPD_TR_SELF_DESTRUCTED) ? OP_DEL : (tr.flags & TRF_STATE_WRITE) ? OP_PUT_ACCOUNT : OP_NONE;
  o.a1 = v.rec_base + tr.rec, o.a2 = tr.txn, o.owner = OWNER_STATE_TRIE;
  v.ops2[tx.op2_begin + rank] = o;
}
// per storage key k of trace t (its slot reads, then its slot writes; with TRF_MIN_KEYS the writes once more under the
// shortened key decoding.rs:235 hashes): its rank among the trace's keys, rlp(U256 value) of a write into val_pool
PPD_HD PPD_INLINE void prep_storage_key(const View& v, uint32_t t, uint32_t k) {
  const TxnTrace& tr = v.traces[t];
  const bool min_keys = (tr.flags & TRF_MIN_KEYS) != 0;
  auto key_of = [&](uint32_t q) -> uint32_t {  // digest index of key q
    if (q < tr.n_reads) return tr.m_reads + q;
    if (q < tr.n_reads + tr.n_writes) return tr.m_wfull + (q - tr.n_reads);
    return tr.m_wmin + (q - tr.n_reads - tr.n_writes);
  };
  auto writes = [&](uint32_t q) -> bool { return min_keys ? q >= tr.n_reads + tr.n_writes : q >= tr.n_reads; };
  const uint32_t mk = key_of(k);
  const uint8_t* me = digest(v, mk);
  uint32_t rank = 0;
  for (uint32_t u = 0; u < tr.n_keys; u++) {
    if (u == k) continue;
    const int c = cmp32(digest(v, key_of(u)), me);
    if (c == 0 && writes(u) && writes(k)) raise(v, TXF_DUP_KEY, tr.txn);  // (a slot may be read and written; written twice it cannot be)
    if (c < 0 || (c == 0 && u < k)) rank++;
  }
  SOp o;
  o.koff = v.dig_base + 32u * mk, o.klen = 64, o.lcp = -1, o.owner = t, o.a1 = o.a2 = 0;
  o.pad = (min_keys && writes(k)) ? 0 : SOP_MARK;  // the shortened key is not one create_trie_subset is given
  o.kind = OP_NONE;
  if (writes(k)) {
    const uint32_t w = k - tr.n_reads - (min_keys ? tr.n_writes : 0);
    const uint8_t* val = v.flat + tr.off_writes + 64ull * w + 32;
    uint32_t z = 0;
    while (z < 32 && val[z] == 0) z++;
    const uint32_t sig = 32 - z;
    if (sig == 0) {  // rlp(0) == [0x80]: a delete (decoding.rs:238-243)
      o.kind = OP_DEL;
    } else {
      uint8_t* dst = v.val_pool + v.val_base + tr.val0 + 36u * w;
      uint32_t el = 0;
      if (sig == 1 && val[31] < 0x80) {
        dst[el++] = val[31];
      } else {
        dst[el++] = (uint8_t)(0x80 + sig);
        for (uint32_t q = 0; q < sig; q++) dst[el++] = val[z + q];
      }
      o.kind = OP_PUT_LEAF, o.a1 = v.val_base + tr.val0 + 36u * w, o.a2 = el;
    }
  }
  v.ops1[tr.op0 + rank] = o;
}
// per txn: the inserts into the transactions and receipts tries (decoding.rs:284-289), after the storage keys; the same
// keys are the ones the tries' subsets are cut with (decoding.rs:190-197)
// (a group of `nthreads` threads per txn: the txn's bytes and its receipt are copied by all of them)
PPD_HD PPD_INLINE void prep_txn(const View& v, uint32_t ti, uint32_t tid = 0, uint32_t nthreads = 1) {
  const TxnDesc& tx = v.txns[ti];
  if (tid == 0) {
    SOp o;
    o.koff = tx.key_off, o.klen = (uint8_t)tx.key_nibs, o.lcp = -1, o.pad = SOP_MARK, o.kind = OP_PUT_LEAF;
    o.a1 = tx.val_txn, o.a2 = tx.len_txn_bytes, o.owner = OWNER_TXN_TRIE;
    v.ops1[tx.op1_end - 2] = o;
    o.a1 = tx.val_receipt, o.a2 = tx.len_receipt, o.owner = OWNER_RECEIPT_TRIE;
    v.ops1[tx.op1_end - 1] = o;
  }
  for (uint32_t k = tid; k < tx.len_txn_bytes; k += nthreads) v.val_pool[tx.val_txn + k] = v.flat[tx.off_txn_bytes + k];
  for (uint32_t k = tid; k < tx.len_receipt; k += nthreads) v.val_pool[tx.val_receipt + k] = v.flat[tx.off_receipt + k];
}
// per sorted key: the LCP with its predecessor in the same trie (state keys carry their txn in a2: one state trie version
// per txn).  Equal keys (a slot read and written) get the full length: the later one then shares everything with the earlier.
PPD_HD PPD_INLINE void prep_lcp(const View& v, SOp* ops, uint32_t i) {
  const bool first = i == 0 || ops[i - 1].owner != ops[i].owner || (ops[i].owner == OWNER_STATE_TRIE && ops[i - 1].a2 != ops[i].a2);
  if (first) {
    ops[i].lcp = -1;
    return;
  }
  const int l = lcp_nibbles(v, ops[i - 1].koff, ops[i - 1].klen, ops[i].koff, ops[i].klen);
  if ((l >= (int)ops[i].klen) != (l >= (int)ops[i - 1].klen)) raise(v, TXF_KEY_PREFIX, 0);
  ops[i].lcp = (int8_t)l;
}

// ---- the account table: slot of every trace's address, initial PartialTrieState entry of every account --------
struct AcctInit {
  uint32_t table_mask;           // slots - 1
  uint32_t state_root;           // root of the pre-image state trie
  const uint32_t* join_storage;  // per pre-image account: root of the storage trie the by-root join gives it, or ST_ABSENT
  const uint32_t* join_root;     // its NK_ROOT node, or NONE
};
PPD_HD PPD_INLINE uint32_t get_leaf(const View& v, uint32_t root, uint32_t koff, uint32_t klen) {
  uint32_t node = root, pos = 0;
  while (node != NODE_EMPTY) {
    if (is_hash_id(node)) return NODE_EMPTY;
    const NodeRec r = v.nodes[node];
    const uint32_t kind = r.w0 & 0xffu, ns = (r.w0 >> 8) & 0xffu, nl = (r.w0 >> 16) & 0xffu;
    if (kind == NK_ROOT) return NODE_EMPTY;
    if (kind == NK_BRANCH) {
      if (pos >= klen) return NODE_EMPTY;
      node = child_at(v, r, key_nib(v, koff, pos));
      pos++;
    } else if (kind == NK_EXT) {
      if (klen - pos < nl || common_prefix(v, r.a0, ns, koff, pos, nl) != nl) return NODE_EMPTY;
      pos += nl;
      node = r.a1;
    } else {
      return (nl == klen - pos && common_prefix(v, r.a0, ns, koff, pos, nl) == nl) ? node : NODE_EMPTY;
    }
  }
  return NODE_EMPTY;
}
PPD_HD PPD_INLINE void acct_claim(const View& v, const AcctInit& a, uint32_t t) {
  const uint8_t* me = digest(v, t);
  uint32_t h = ((uint32_t)me[4] | ((uint32_t)me[5] << 8) | ((uint32_t)me[6] << 16) | ((uint32_t)me[7] << 24)) & a.table_mask;
  for (;;) {
    const uint32_t prev = PPD_ATOMIC_CAS(&v.acct[h].owner, 0xffffffffu, t);
    if (prev == 0xffffffffu) {
      // first trace of this address: the account's entry in the initial PartialTrieState
      AcctState s;
      s.owner = t, s.storage = ST_ABSENT, s.root_node = NONE, s.pre_rec = NONE;
      const uint32_t leaf = get_leaf(v, a.state_root, v.dig_base + 32u * t, 64);
      if (leaf != NODE_EMPTY && (v.nodes[leaf].w0 & 0xffu) == NK_LEAF_ACCOUNT) {
        const uint32_t r = v.nodes[leaf].a1;
        s.pre_rec = r, s.storage = a.join_storage[r], s.root_node = a.join_root[r];
        v.pre_slot[r] = h;
      }
      v.acct[h].storage = s.storage, v.acct[h].root_node = s.root_node, v.acct[h].pre_rec = s.pre_rec;
      v.traces[t].acct = h;
      return;
    }
    if (prev == t || cmp32(digest(v, prev), me) == 0) {
      v.traces[t].acct = h;
      return;
    }
    h = (h + 1) & a.table_mask;
  }
}

// ---- the by-address join of a direct pre-image (kind 2, host_direct.cu) -------------------------------------------
// The storage map of a Separate pre-image is keyed by hashed address: an account has a storage trie iff its address is
// in the map, and then it is the trie sent for it (its own, in the re-spelled witness).  This is the map the host path
// builds (build_pre_image, then direct_filter_storage), account by account:
//   not in the map                      ST_ABSENT / NONE, even when its root is that of a trie in the map
//   in the map, trie not empty          its own trie (a bare hash node included) and its NK_ROOT node
//   in the map, trie empty (its root is EMPTY_TRIE_HASH: an empty trie, or a hash node of that root)
//                                       the empty-rooted trie witnessed LAST (the host builder's empty form) / NONE
// Every account keeps a trie of its own or the empty form, so this join never shares an expanded trie.
PPD_HD PPD_INLINE uint32_t addr_slot_hash(const uint8_t* k, uint32_t mask) {
  return ((uint32_t)k[8] | ((uint32_t)k[9] << 8) | ((uint32_t)k[10] << 16) | ((uint32_t)k[11] << 24)) & mask;
}
PPD_HD PPD_INLINE bool eq32(const uint8_t* a, const uint8_t* b) {
  bool same = true;
  for (int i = 0; i < 32; i++) same &= a[i] == b[i];
  return same;
}
// thread i: map entry i into the table; account i, if its witnessed storage trie is empty, into the empty-form cell
PPD_HD PPD_INLINE void join_addr_insert(const JoinView& j, uint32_t i) {
  if (i < j.n_acct && (j.acct_list[5ull * i + 3] & 3u) == 1u) PPD_ATOMIC_MAX(&j.slot_best[0], i + 1u);
  if (i >= j.n_keep) return;
  const uint8_t* key = j.keep + 32ull * i;
  uint32_t h = addr_slot_hash(key, j.table_mask);
  for (;;) {
    const uint32_t prev = PPD_ATOMIC_CAS(&j.slot_owner[h], 0xffffffffu, i);
    if (prev == 0xffffffffu || eq32(j.keep + 32ull * prev, key)) return;  // (the map has no duplicates: host_direct.cu)
    h = (h + 1) & j.table_mask;
  }
}
// account r: its hashed address from its leaf key, right-aligned as export_account assembles it (utils.rs:49-59)
PPD_HD PPD_INLINE void join_addr_resolve(const View& v, const JoinView& j, uint32_t r) {
  const uint32_t* al = j.acct_list + 5ull * r;
  const NodeRec nr = v.nodes[al[0]];
  const uint32_t ns = (nr.w0 >> 8) & 0xffu, nl = (nr.w0 >> 16) & 0xffu, klen = ns + nl;
  uint8_t haddr[32];
  for (int i = 0; i < 32; i++) haddr[i] = 0;
  for (uint32_t k = 0; k < klen && k < 64; k++) {
    const uint32_t posn = 64 - klen + k, nib = key_nib(v, nr.a0, k);
    haddr[posn >> 1] |= (uint8_t)((posn & 1) ? nib : (nib << 4));
  }
  const uint32_t flags = al[3];
  j.pre_flags[r] = (uint8_t)((flags >> 1) & 1u);
  uint32_t storage = ST_ABSENT, root = NONE;
  for (uint32_t h = addr_slot_hash(haddr, j.table_mask);; h = (h + 1) & j.table_mask) {
    const uint32_t own = j.slot_owner[h];
    if (own == 0xffffffffu) break;
    if (!eq32(j.keep + 32ull * own, haddr)) continue;
    if (flags & 2u) {
      storage = al[1], root = al[2] == NODE_EMPTY ? NONE : al[2];
    } else {
      const uint32_t last = j.slot_best[0];
      if (last) storage = j.acct_list[5ull * (last - 1u) + 1];
    }
    break;
  }
  j.join_storage[r] = storage, j.join_root[r] = root;
}

// ---- the loop itself: one thread block per block of txns (the harness runs it as a block of one thread) ------
#if defined(__CUDA_ARCH__)
#define PPD_BLOCK_SYNC() __syncthreads()
#define PPD_PHASE_CLOCK(c, k)                                \
  do {                                                       \
    if ((c).tid == 0) {                                      \
      const long long now_ = clock64();                      \
      (c).v.cur->phase_clocks[k] += now_ - *(c).sh_clock;    \
      *(c).sh_clock = now_;                                  \
    }                                                        \
  } while (0)
#else
#define PPD_BLOCK_SYNC() ((void)0)
#define PPD_PHASE_CLOCK(c, k) ((void)0)
#endif

PPD_HD PPD_INLINE void copy32(uint8_t* d, const uint8_t* s) {
  for (int i = 0; i < 32; i++) d[i] = s[i];
}

PPD_HD PPD_INLINE void run_txn(const Ctx& c, uint32_t ti, const uint8_t* empty_trie_hash, const uint8_t* empty_code_hash) {
  const View& v = c.v;
  const TxnDesc tx = v.txns[ti];
  const uint32_t ntr = tx.trace_end - tx.trace_begin;
  const uint32_t n1 = tx.op1_end - tx.op1_begin, n2 = tx.op2_end - tx.op2_begin;
  // the txn's keys: in shared memory next to the scratch when they fit
  const SOp* ops1 = v.ops1 + tx.op1_begin;
  const SOp* ops2 = v.ops2 + tx.op2_begin;
  if (SCR(v).sh_ops) {
    for (uint32_t k = c.tid; k < n1 + n2; k += c.nthreads) SCR(v).sh_ops[k] = k < n1 ? ops1[k] : ops2[k - n1];
    ops1 = SCR(v).sh_ops, ops2 = SCR(v).sh_ops + n1;
  }
  // ---- the tries the subsets are cut from (decoding.rs:179-217): roots before the txn ----
  if (c.tid == 0) {
    v.seg_b[tx.seg_tries + 0] = v.cur->state_root;
    v.seg_b[tx.seg_tries + 1] = v.cur->txn_root;
    v.seg_b[tx.seg_tries + 2] = v.cur->receipt_root;
    *SCR(v).pc_count = 0;
  }
  for (uint32_t k = c.tid; k <= SCR(v).pc_map_mask; k += c.nthreads) SCR(v).pc_map_key[k] = 0xffffffffu;
  for (uint32_t k = c.tid; k < ntr; k += c.nthreads) {
    const uint32_t t = tx.trace_begin + k;
    const TxnTrace& tr = v.traces[t];
    AcctState& a = v.acct[tr.acct];
    if (a.storage == ST_ABSENT) {
      // a missing storage trie: Hash(pre-image storage root) when the account had storage in the pre-image and this txn
      // does not access its slots, else an empty trie (decoding.rs:572-582); it stays in the live state
      uint32_t s = NODE_EMPTY;
      if (a.pre_rec != NONE && (v.pre_flags[a.pre_rec] & 1u) && tr.n_reads + tr.n_writes == 0) s = v.accounts[a.pre_rec].storage_src;
      a.storage = s, a.root_node = NONE;
    }
    v.seg_a[tx.seg_storage + 2 * tr.rank] = v.dig_base + 32u * t;
    v.seg_b[tx.seg_storage + 2 * tr.rank] = IR_SEG_KEY32;
    v.seg_a[tx.seg_storage + 2 * tr.rank + 1] = 0;
    v.seg_b[tx.seg_storage + 2 * tr.rank + 1] = a.storage;
  }
  PPD_BLOCK_SYNC();
  PPD_PHASE_CLOCK(c, 0);
  if (c.tid == 0) PPD_EV(v, ti, 0, 100 + 0);
  // ---- every key of the txn walks the tries as they are before the txn: the marking walks of
  // create_minimal_partial_tries_needed_by_txn (decoding.rs:179-217) and the first half of the writes ----
  const Batch b1{ops1, n1, 0, ti}, b2{ops2, n2, n1, ti};
  for (uint32_t k = c.tid; k < n1 + n2; k += c.nthreads) {
    uint32_t* out = v.touched + tx.touched_base + MARK_SLOTS_T * k;
    if (k < n1)
      batch_walk(c, b1, k, out);
    else
      batch_walk(c, b2, k - n1, out);
  }
  PPD_BLOCK_SYNC();
  PPD_PHASE_CLOCK(c, 1);
  if (c.tid == 0) PPD_EV(v, ti, 0, 100 + 1);
  {
    const uint32_t n_pc = *SCR(v).pc_count < SCR(v).pc_n_fast + SCR(v).pc_n_slow ? *SCR(v).pc_count : SCR(v).pc_n_fast + SCR(v).pc_n_slow;
    for (uint32_t k = c.tid; k < n_pc; k += c.nthreads) {
      PPD_EV(v, ti, c.tid, 3);
      pc_fill(v, k);
      PPD_EV(v, ti, c.tid, 4);
    }
  }
  for (uint32_t k = c.tid; k < n1 + n2; k += c.nthreads) {
    PPD_EV(v, ti, c.tid, 5);
    if (k < n1)
      batch_announce(c, b1, k);
    else
      batch_announce(c, b2, k - n1);
    PPD_EV(v, ti, c.tid, 6);
  }
  PPD_BLOCK_SYNC();
  PPD_PHASE_CLOCK(c, 2);
  if (c.tid == 0) PPD_EV(v, ti, 0, 100 + 2);
  // ---- apply_deltas_to_trie_state (decoding.rs:219-292): storage writes, the txn and receipt inserts ----
  for (uint32_t k = c.tid; k < n1; k += c.nthreads) {
    PPD_EV(v, ti, c.tid, 10);
    batch_climb(c, b1, k);
    PPD_EV(v, ti, c.tid, 14);
  }
  PPD_BLOCK_SYNC();
  PPD_PHASE_CLOCK(c, 3);
  if (c.tid == 0) PPD_EV(v, ti, 0, 100 + 3);
  // ---- the accounts after the txn: storage_root = the storage trie's hash after the writes (late-bound: an NK_ROOT node) ----
  for (uint32_t k = c.tid; k < ntr; k += c.nthreads) {
    PPD_EV(v, ti, c.tid, 30);
    const uint32_t t = tx.trace_begin + k;
    const TxnTrace& tr = v.traces[t];
    if (!(tr.flags & TRF_STATE_WRITE)) continue;
    AccountRec rec;
    const uint32_t e = n1 + tr.rank;  // the trace's state key: its walk found the account as state.get() would (decoding.rs:251-254)
    if (SCR(v).tkind[e] == TK_LEAF_SAME) {
      const uint32_t leaf = SCR(v).tnode[e];
      if ((v.nodes[leaf].w0 & 0xffu) != NK_LEAF_ACCOUNT) {
        raise(v, TXF_NOT_ACCOUNT, ti);
        continue;
      }
      rec = v.accounts[v.nodes[leaf].a1];
    } else {  // EMPTY_ACCOUNT_BYTES_RLPED
      for (int i = 0; i < 32; i++) rec.nonce[i] = 0, rec.balance[i] = 0;
      copy32(rec.storage_root, empty_trie_hash);
      copy32(rec.code_hash, empty_code_hash);
      rec.storage_src = NODE_EMPTY;
      rec.pad[0] = rec.pad[1] = rec.pad[2] = 0;
    }
    if (tr.n_writes) {
      AcctState& a = v.acct[tr.acct];
      if (a.root_node == NONE) a.root_node = new_root(v, a.storage);
      rec.storage_src = a.root_node;
    }
    if (tr.flags & PPD_TR_BALANCE) copy32(rec.balance, v.flat + tr.off_balance);
    if (tr.flags & PPD_TR_NONCE) copy32(rec.nonce, v.flat + tr.off_nonce);
    if (tr.flags & PPD_TR_CODE_READ)
      copy32(rec.code_hash, v.flat + tr.code_off);
    else if (tr.flags & PPD_TR_CODE_WRITE)
      copy32(rec.code_hash, digest(v, tr.m_code));
    v.accounts[v.rec_base + tr.rec] = rec;
    PPD_EV(v, ti, c.tid, 31);
  }
  PPD_BLOCK_SYNC();  // (a new account leaf's level follows from its record's storage root node: new_leaf_for)
  PPD_PHASE_CLOCK(c, 4);
  if (c.tid == 0) PPD_EV(v, ti, 0, 100 + 4);
  // ---- state writes and self-destructs in one descent ----
  for (uint32_t k = c.tid; k < n2; k += c.nthreads) {
    PPD_EV(v, ti, c.tid, 20);
    batch_climb(c, b2, k);
    PPD_EV(v, ti, c.tid, 24);
  }
  PPD_BLOCK_SYNC();
  PPD_PHASE_CLOCK(c, 5);
  if (c.tid == 0) PPD_EV(v, ti, 0, 100 + 5);
  for (uint32_t k = c.tid; k < ntr; k += c.nthreads) {
    const TxnTrace& tr = v.traces[tx.trace_begin + k];
    if (tr.flags & PPD_TR_SELF_DESTRUCTED) {  // trie_state.storage.remove(hashed_addr), decoding.rs:271-282
      AcctState& a = v.acct[tr.acct];
      a.storage = ST_ABSENT, a.root_node = NONE;
    }
  }
  // ---- calculate_trie_input_hashes (decoding.rs:458-464): three NK_ROOT nodes, read by the dump as refs ----
  if (c.tid == 0) {
    v.seg_a[tx.seg_roots + 0] = new_root(v, v.cur->state_root);
    v.seg_a[tx.seg_roots + 1] = new_root(v, v.cur->txn_root);
    v.seg_a[tx.seg_roots + 2] = new_root(v, v.cur->receipt_root);
  }
  PPD_BLOCK_SYNC();
  PPD_PHASE_CLOCK(c, 6);
  if (c.tid == 0) PPD_EV(v, ti, 0, 100 + 6);
}

// ---- after the last txn: the NK_ROOT nodes dummy entries refer to, and the withdrawals (decoding.rs:356-428) ----
PPD_HD PPD_INLINE void u256_add(uint8_t* a, const uint8_t* b) {
  uint32_t carry = 0;
  for (int i = 31; i >= 0; i--) {
    const uint32_t x = (uint32_t)a[i] + b[i] + carry;
    a[i] = (uint8_t)x;
    carry = x >> 8;
  }
}
PPD_HD PPD_INLINE void run_finish(const Ctx& c, uint32_t initial_state) {
  const View& v = c.v;
  if (c.tid == 0 && !v.cur->flag) {
    Cursors& cur = *v.cur;
    cur.roots[XR_INITIAL_STATE] = new_root(v, initial_state);
    cur.roots[XR_EMPTY] = new_root(v, NODE_EMPTY);
    cur.roots[XR_FINAL_STATE] = new_root(v, cur.state_root);
    cur.roots[XR_FINAL_TXN] = new_root(v, cur.txn_root);
    cur.roots[XR_FINAL_RECEIPT] = new_root(v, cur.receipt_root);
    cur.state_before_withdrawals = cur.state_root;
    // one after the other, as the reference does: a later withdrawal to the same address sees the earlier one
    for (uint32_t w = 0; w < v.n_withdrawals && !cur.flag; w++) {
      const Withdrawal wd = v.withdrawals[w];
      const uint32_t koff = v.dig_base + 32u * wd.m_addr;
      const uint32_t leaf = get_leaf(v, cur.state_root, koff, 64);
      if (leaf == NODE_EMPTY || (v.nodes[leaf].w0 & 0xffu) != NK_LEAF_ACCOUNT) {
        raise(v, TXF_WITHDRAWAL, 0xffffffffu);
        break;
      }
      AccountRec rec = v.accounts[v.nodes[leaf].a1];
      u256_add(rec.balance, v.flat + wd.off_amount);
      v.accounts[v.rec_base + wd.rec] = rec;
      SOp o;
      o.koff = koff, o.klen = 64, o.lcp = -1, o.kind = OP_PUT_ACCOUNT, o.pad = 0, o.a1 = v.rec_base + wd.rec, o.a2 = 0, o.owner = OWNER_STATE_TRIE;
      cur.state_root = insert_one(v, NL{cur.state_root, lvl(v, cur.state_root)}, 0, o, 0xffffffffu).id;
    }
    cur.roots[XR_AFTER_WITHDRAWALS] = new_root(v, cur.state_root);
  }
  PPD_BLOCK_SYNC();
}

// ---- the storage map for dummy entries (decoding.rs:531-549 lists EVERY storage trie): per pre-image account its
// hashed address and the root of its trie before the first and after the last txn ----
struct AcctExport {
  uint8_t haddr[32];
  uint32_t initial, final_;  // node id, NODE_EMPTY, or ST_ABSENT
};
PPD_HD PPD_INLINE void export_account(const View& v, const uint32_t* acct_list, const uint32_t* join_storage, uint32_t r, AcctExport* out) {
  const NodeRec nr = v.nodes[acct_list[5ull * r]];
  const uint32_t ns = (nr.w0 >> 8) & 0xffu, nl = (nr.w0 >> 16) & 0xffu, klen = ns + nl;
  AcctExport e;
  for (int i = 0; i < 32; i++) e.haddr[i] = 0;
  for (uint32_t k = 0; k < klen && k < 64; k++) {  // utils.rs:49-59: the nibbles right-aligned in 32 bytes
    const uint32_t posn = 64 - klen + k, nib = key_nib(v, nr.a0, k);
    e.haddr[posn >> 1] |= (uint8_t)((posn & 1) ? nib : (nib << 4));
  }
  e.initial = join_storage[r];
  const uint32_t slot = v.pre_slot[r];
  e.final_ = slot < NONE ? v.acct[slot].storage : e.initial;
  out[r] = e;
}

}  // namespace txn
}  // namespace ppd
