// ppd_txn.cu — the txn loop on the GPU: kernels around txn_core.h.
//
//   txn_msgs_kernel      byte ranges of the FlatBlock to hash (addresses, slot keys, written code), one thread per trace
//   join_*_kernel        convert_storage_trie_root_keyed_hashmap_to_account_addr_keyed (compact_to_partial_trie.rs:167-190):
//                        accounts get the storage trie witnessed LAST under their storage root, whoever witnessed it
//   join_addr_*_kernel   the same for a direct pre-image, whose storage map is by hashed address (txn_core.h)
//   acct_claim_kernel    one table slot per distinct address; the account's entry in the initial PartialTrieState
//   prep_*_kernel        ops of every txn sorted per trie (rank sort: batches are tens of keys, O(n^2) is parallel and tiny),
//                        written values RLP-encoded into val_pool, LCPs of neighbours
//   txn_loop_kernel      ONE thread block runs the whole txn loop of a block (decoding.rs:80-177): txns are sequential,
//                        the keys of a txn parallel; blocks of a batch run concurrently, one lane each
// All of it is pointer chasing over the arena: latency bound by construction (a walk is ~2 dependent loads per trie
// level), which is why a block's loop is one resident CTA that other lanes' kernels overlap, not a grid.
#include <cstdint>
#include <cstdlib>

#include "ppd_kernels.h"
#include "txn_core.h"

namespace ppd {

using namespace txn;

namespace {

__constant__ uint8_t C_EMPTY_TRIE[32] = {0x56, 0xe8, 0x1f, 0x17, 0x1b, 0xcc, 0x55, 0xa6, 0xff, 0x83, 0x45, 0xe6, 0x92, 0xc0, 0xf8, 0x6e,
                                         0x5b, 0x48, 0xe0, 0x1b, 0x99, 0x6c, 0xad, 0xc0, 0x01, 0x62, 0x2f, 0xb5, 0xe3, 0x63, 0xb4, 0x21};
__constant__ uint8_t C_EMPTY_CODE[32] = {0xc5, 0xd2, 0x46, 0x01, 0x86, 0xf7, 0x23, 0x3c, 0x92, 0x7e, 0x7d, 0xb2, 0xdc, 0xc7, 0x03, 0xc0,
                                         0xe5, 0x00, 0xb6, 0x53, 0xca, 0x82, 0x27, 0x3b, 0x7b, 0xfa, 0xd8, 0x04, 0x5d, 0x85, 0xa4, 0x70};

__global__ void txn_msgs_kernel(View v, uint64_t* __restrict__ se) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < v.n_traces) prep_msgs(v, t, se);
  if (t < v.n_withdrawals) prep_withdrawal_msg(v, t, se);
}

__global__ void txn_init_kernel(View v, Cursors init, uint32_t table_slots) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *v.cur = init;
  if (i < table_slots) v.acct[i] = AcctState{ST_ABSENT, NONE, NONE, 0xffffffffu};
  // (pre_slot[] is reset by the launcher's memset)
}

// ---- the by-root join ------------------------------------------------------------------------------------
__device__ __forceinline__ const uint8_t* storage_root_of(const JoinView& j, uint32_t r) {
  const uint32_t flags = j.acct_list[5ull * r + 3];
  return (flags & 2u) ? j.ref + 32ull * j.acct_list[5ull * r + 2] : C_EMPTY_TRIE;
}
__device__ __forceinline__ bool same32(const uint8_t* a, const uint8_t* b) {
  bool same = true;
  for (int i = 0; i < 32; i++) same &= a[i] == b[i];
  return same;
}
__device__ __forceinline__ uint32_t root_slot_hash(const uint8_t* k, uint32_t mask) {
  return ((uint32_t)k[8] | ((uint32_t)k[9] << 8) | ((uint32_t)k[10] << 16) | ((uint32_t)k[11] << 24)) & mask;
}
// every account that witnesses a storage node: the table entry of its root keeps the LAST such account
__global__ void join_insert_kernel(JoinView j) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= j.n_acct) return;
  if (!(j.acct_list[5ull * r + 3] & 1u)) return;
  const uint8_t* key = storage_root_of(j, r);
  uint32_t h = root_slot_hash(key, j.table_mask);
  for (;;) {
    const uint32_t prev = atomicCAS(&j.slot_owner[h], 0xffffffffu, r);
    if (prev == 0xffffffffu || prev == r || same32(storage_root_of(j, prev), key)) {
      atomicMax(&j.slot_best[h], r + 1u);
      return;
    }
    h = (h + 1) & j.table_mask;
  }
}
__global__ void join_resolve_kernel(JoinView j) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= j.n_acct) return;
  const uint8_t* key = storage_root_of(j, r);
  j.pre_flags[r] = (uint8_t)((j.acct_list[5ull * r + 3] >> 1) & 1u);
  uint32_t h = root_slot_hash(key, j.table_mask), storage = ST_ABSENT, root = NONE;
  for (;;) {
    const uint32_t own = j.slot_owner[h];
    if (own == 0xffffffffu) break;
    if (same32(storage_root_of(j, own), key)) {
      const uint32_t best = j.slot_best[h] - 1u;
      storage = j.acct_list[5ull * best + 1];
      root = j.acct_list[5ull * best + 2];
      if (root == NODE_EMPTY) root = NONE;
      // another account's expanded trie: the reference clones it (compact_to_partial_trie.rs:183-185), because a
      // txn that touches both accounts cuts a separate subset out of each; the host path does that
      if (best != r && storage < HASH_BASE) atomicCAS(j.flag, 0u, (uint32_t)TXF_SHARED_TRIE);
      break;
    }
    h = (h + 1) & j.table_mask;
  }
  j.join_storage[r] = storage, j.join_root[r] = root;
}

// ---- the by-address join (direct pre-images; txn_core.h: join_addr_insert / join_addr_resolve) -------------------
__global__ void join_addr_insert_kernel(JoinView j, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) join_addr_insert(j, i);
}
__global__ void join_addr_resolve_kernel(View v, JoinView j) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < j.n_acct) join_addr_resolve(v, j, r);
}

__global__ void acct_claim_kernel(View v, AcctInit a) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < v.n_traces) acct_claim(v, a, t);
}
__global__ void prep_trace_kernel(View v) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < v.n_traces) prep_trace(v, t);
}
// grid (trace, chunk of its storage keys)
__global__ void prep_storage_key_kernel(View v) {
  const uint32_t t = blockIdx.x, k = blockIdx.y * blockDim.x + threadIdx.x;
  if (k < v.traces[t].n_keys) prep_storage_key(v, t, k);
}
__global__ void prep_txn_kernel(View v) {
  prep_txn(v, blockIdx.x, threadIdx.x, blockDim.x);  // one thread block per txn
}
__global__ void prep_lcp_kernel(View v, uint32_t n1, uint32_t n2) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n1)
    prep_lcp(v, v.ops1, i);
  else if (i < n1 + n2)
    prep_lcp(v, v.ops2, i - n1);
}

__global__ void acct_export_kernel(View v, const uint32_t* __restrict__ acct_list, const uint32_t* __restrict__ join_storage, uint32_t n_acct,
                                   AcctExport* __restrict__ out) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n_acct) export_account(v, acct_list, join_storage, r, out);
}

constexpr int LOOP_THREADS = 256;
constexpr uint32_t LOOP_SCRATCH_BYTES = (sizeof(Scratch) + 15) & ~15u;
constexpr uint32_t SH_KEYS = 512;   // keys of one txn whose scratch fits in shared memory
#ifndef PPD_SH_NODES
#define PPD_SH_NODES 384
#define PPD_SH_MAP 2048
#endif
constexpr uint32_t SH_NODES = PPD_SH_NODES;  // path-node table entries in shared memory (the rest of a txn's spill to HBM)
constexpr uint32_t SH_MAP = PPD_SH_MAP;   // slots of the node id -> entry map
struct LoopShared {
  PathNode pc[SH_NODES];
  uint32_t path_node[SH_KEYS * PATH_CAP], path_pc[SH_KEYS * PATH_CAP];
  uint32_t pc_map[SH_MAP], pc_map_key[SH_MAP];
  uint32_t tnode[SH_KEYS], tpc[SH_KEYS], key_hi[SH_KEYS];
  SOp ops[SH_KEYS];
  uint8_t path_depth[SH_KEYS * PATH_CAP];
  uint8_t plen[SH_KEYS], tdepth[SH_KEYS], tkind[SH_KEYS];
};
// txns [ti0, ti1) of the block.  The loop of a block is launched in chunks so that the kernels of another lane that
// shares the hardware queue (the device has at most 32 of them) are not held up behind one long kernel.  use_shared: the
// scratch of a txn (path, terminal, result per key) and its keys live in shared memory: every step of the re-assembly
// then costs one trip to L2 / HBM (the child table) instead of four.
struct LoopBatchArg {
  LoopTask t[LOOP_BATCH_MAX];
};
// One thread block per task (= per block of the batch): blocks of different lanes whose loops are due together run as
// one launch (gpu_txn.cu: LoopBatcher), so a loop does not hold a lane's stream (one of the device's 32 hardware queues)
// for its whole length.  tasks: device-accessible (page-locked host memory), read once per launch.
__global__ void __launch_bounds__(LOOP_THREADS, 1) txn_loop_kernel(const __grid_constant__ LoopBatchArg A, uint32_t ti0, uint32_t ti1) {
  extern __shared__ __align__(16) uint8_t loop_smem[];  // [Scratch | LoopShared when the txns' keys fit]
  __shared__ uint32_t sh_stop, sh_cursor[4], sh_pc_count;
  __shared__ long long sh_clock;
  const View& v = A.t[blockIdx.x].v;  // (kernel-parameter space: fields are read from the constant bank)
  const uint32_t initial_state = A.t[blockIdx.x].initial_state, use_shared = A.t[blockIdx.x].use_shared;
  if (ti1 > v.n_txns) ti1 = v.n_txns;
  if (ti0 > ti1 || (ti0 == ti1 && ti0 != 0)) return;  // this block's txns ended in an earlier launch of the batch
  const bool finish = ti1 == v.n_txns;
  if (threadIdx.x == 0) {
    sh_clock = clock64();
    sh_cursor[0] = v.cur->n_nodes, sh_cursor[1] = v.cur->n_children, sh_cursor[2] = v.cur->key_bytes, sh_cursor[3] = v.cur->max_level;
    sh_stop = *reinterpret_cast<volatile uint32_t*>(&v.cur->flag);
    Scratch sc = v.s;
    sc.a_nodes = &sh_cursor[0], sc.a_children = &sh_cursor[1], sc.a_keys = &sh_cursor[2], sc.a_max_level = &sh_cursor[3];
    if (use_shared) {
      LoopShared& S = *reinterpret_cast<LoopShared*>(loop_smem + LOOP_SCRATCH_BYTES);
      sc.path_node = S.path_node, sc.path_pc = S.path_pc, sc.path_depth = S.path_depth;
      sc.plen = S.plen, sc.tnode = S.tnode, sc.tpc = S.tpc, sc.tdepth = S.tdepth, sc.tkind = S.tkind, sc.key_hi = S.key_hi, sc.sh_ops = S.ops;
      sc.pc_fast = S.pc, sc.pc_n_fast = SH_NODES, sc.pc_map = S.pc_map, sc.pc_map_key = S.pc_map_key, sc.pc_map_mask = SH_MAP - 1;
      // (pc_slow / pc_n_slow: the HBM tier the host laid out; a txn with more path nodes than the map takes is flagged)
      if (sc.pc_n_slow > SH_MAP / 2 - SH_NODES) sc.pc_n_slow = SH_MAP / 2 - SH_NODES;
    }
    sc.pc_count = &sh_pc_count;
#if defined(__CUDA_ARCH__)
    SCR(v) = sc;
#endif
  }
  __syncthreads();
  if (sh_stop) return;  // an earlier chunk (or the join) raised a flag: the host path redoes the block
  Ctx c{v, threadIdx.x, blockDim.x, &sh_clock};
  for (uint32_t ti = ti0; ti < ti1; ti++) {
    run_txn(c, ti, C_EMPTY_TRIE, C_EMPTY_CODE);
    // a raised flag ends the loop; one thread reads it so that the decision is uniform
    if (threadIdx.x == 0) sh_stop = *reinterpret_cast<volatile uint32_t*>(&v.cur->flag);
    __syncthreads();
    if (sh_stop) break;
    __syncthreads();
  }
  if (finish) run_finish(c, initial_state);
  __syncthreads();
  if (threadIdx.x == 0) v.cur->n_nodes = sh_cursor[0], v.cur->n_children = sh_cursor[1], v.cur->key_bytes = sh_cursor[2], v.cur->max_level = sh_cursor[3];
}

}  // namespace

static inline uint32_t cdiv(uint32_t a, uint32_t b) { return (a + b - 1) / b; }

void launch_txn_msgs(const View& v, uint64_t* se, cudaStream_t st) {
  const uint32_t n = v.n_traces > v.n_withdrawals ? v.n_traces : v.n_withdrawals;
  if (n) txn_msgs_kernel<<<cdiv(n, 128), 128, 0, st>>>(v, se);
}
void launch_txn_init(const View& v, const Cursors& init, uint32_t table_slots, cudaStream_t st) {
  txn_init_kernel<<<cdiv(table_slots, 256), 256, 0, st>>>(v, init, table_slots);
}
void launch_join(const JoinView& j, cudaStream_t st) {
  if (!j.n_acct) return;
  join_insert_kernel<<<cdiv(j.n_acct, 128), 128, 0, st>>>(j);
  join_resolve_kernel<<<cdiv(j.n_acct, 128), 128, 0, st>>>(j);
}
void launch_join_by_address(const View& v, const JoinView& j, cudaStream_t st) {
  if (!j.n_acct) return;
  const uint32_t n = j.n_keep > j.n_acct ? j.n_keep : j.n_acct;
  join_addr_insert_kernel<<<cdiv(n, 128), 128, 0, st>>>(j, n);
  join_addr_resolve_kernel<<<cdiv(j.n_acct, 128), 128, 0, st>>>(v, j);
}
uint32_t launch_txn_prep(const View& v, const AcctInit& a, uint32_t n_ops1, uint32_t n_ops2, uint32_t max_writes, cudaStream_t st) {
  uint32_t launches = 0;
  if (v.n_traces) {
    acct_claim_kernel<<<cdiv(v.n_traces, 128), 128, 0, st>>>(v, a);
    prep_trace_kernel<<<cdiv(v.n_traces, 128), 128, 0, st>>>(v);
    launches += 2;
    if (max_writes) {
      const uint32_t threads = max_writes >= 64 ? 128 : 32;
      prep_storage_key_kernel<<<dim3(v.n_traces, cdiv(max_writes, threads)), threads, 0, st>>>(v);
      launches++;
    }
  }
  if (v.n_txns) {
    prep_txn_kernel<<<v.n_txns, 128, 0, st>>>(v);
    prep_lcp_kernel<<<cdiv(n_ops1 + n_ops2, 128), 128, 0, st>>>(v, n_ops1, n_ops2);
    launches += 2;
  }
  return launches;
}
// txns per launch of the loop kernel: a raised flag stops the batch at the next launch.  64 gave 615 blocks/s in a sweep
// (profiles/r02b_knobs.txt: 512 config-2 blocks per stream call), within two runs of 16 at 578 and 617.
constexpr uint32_t LOOP_CHUNK = 16;
uint32_t txn_loop_uses_shared(uint32_t max_keys) { return max_keys <= SH_KEYS ? 1u : 0u; }  // max_keys: the most keys any txn of the block has
uint32_t launch_txn_loops(const LoopTask* tasks, uint32_t n, uint32_t max_txns, bool any_shared, cudaStream_t st) {
  static const bool attr = [] {
    cudaFuncSetAttribute(txn_loop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(LOOP_SCRATCH_BYTES + sizeof(LoopShared)));
    return true;
  }();
  (void)attr;
  const size_t smem = LOOP_SCRATCH_BYTES + (any_shared ? sizeof(LoopShared) : 0);
  if (n > LOOP_BATCH_MAX) n = LOOP_BATCH_MAX;
  static thread_local LoopBatchArg A;  // (copied into the launch: the caller's array is free again on return)
  for (uint32_t k = 0; k < n; k++) A.t[k] = tasks[k];
  uint32_t launches = 0;
  for (uint32_t t0 = 0; t0 < max_txns || launches == 0; t0 += LOOP_CHUNK) {
    txn_loop_kernel<<<n, LOOP_THREADS, smem, st>>>(A, t0, t0 + LOOP_CHUNK);
    launches++;
  }
  return launches;
}
uint32_t launch_txn_loop(LoopTask* slot, const View& v, uint32_t initial_state, uint32_t max_keys, cudaStream_t st) {
  slot->v = v, slot->initial_state = initial_state, slot->use_shared = txn_loop_uses_shared(max_keys);
  return launch_txn_loops(slot, 1, v.n_txns, slot->use_shared != 0, st);
}
void launch_acct_export(const View& v, const JoinView& j, AcctExport* out, cudaStream_t st) {
  if (j.n_acct) acct_export_kernel<<<cdiv(j.n_acct, 128), 128, 0, st>>>(v, j.acct_list, j.join_storage, j.n_acct, out);
}

}  // namespace ppd
