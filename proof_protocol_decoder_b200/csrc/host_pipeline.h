// host_pipeline.h — types shared by the host-side sources of libppd_b200.so: the context and its lanes, the
// views of one block being decoded (FlatBlock reader, witness instruction list, IR plans) and the job that
// owns the page-locked pools.  The sources:
//   ppd_host.cu       context, lanes, key hashing, the sweep, the block pipeline and the C ABI
//   host_witness.cu   compact witness parser + host builder of the pre-image tries (declined witnesses)
//   host_txn.cu       FlatBlock reader, RLP helpers, the host txn loop (shape_block)
//   host_dump.cu      host serialisation of IrDump
//   gpu_pre_image.cu  witness parse + pre-image arena on the GPU (ppd_parse.cu kernels)
//   gpu_dump.cu       IrDump serialisation on the GPU (ppd_dump.cu kernels)
//   gpu_txn.cu        the txn loop on the GPU (ppd_txn.cu kernels)
//   gpu_trie.cu       tries from leaves (ppd_build.cu, ppd_leaves.cu, ppd_subset.cu, ppd_update.cu kernels): the root and
//                     subset entries and the resident trie handles
// The host never computes a Keccak or a node encoding; there is no CPU fallback.
#pragma once
#include <cuda_runtime.h>
#include <sys/mman.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_set>
#include <unordered_map>
#include <vector>

#include "../../include/ppd_b200.h"
#include "arena.h"
#include "devbuf.h"
#include "flat_maps.h"
#include "host_arena.h"
#include "ppd_kernels.h"
#include "txn_tables.h"

namespace ppd {

static const uint8_t EMPTY_CODE_HASH[32] = {0xc5, 0xd2, 0x46, 0x01, 0x86, 0xf7, 0x23, 0x3c, 0x92, 0x7e, 0x7d, 0xb2, 0xdc, 0xc7, 0x03, 0xc0,
                                            0xe5, 0x00, 0xb6, 0x53, 0xca, 0x82, 0x27, 0x3b, 0x7b, 0xfa, 0xd8, 0x04, 0x5d, 0x85, 0xa4, 0x70};
static const uint8_t EMPTY_TRIE_HASH[32] = {0x56, 0xe8, 0x1f, 0x17, 0x1b, 0xcc, 0x55, 0xa6, 0xff, 0x83, 0x45, 0xe6, 0x92, 0xc0, 0xf8, 0x6e,
                                            0x5b, 0x48, 0xe0, 0x1b, 0x99, 0x6c, 0xad, 0xc0, 0x01, 0x62, 0x2f, 0xb5, 0xe3, 0x63, 0xb4, 0x21};

struct Job;
void job_delete(Job*);
void* pinned_alloc(size_t n);
void pinned_free(void* p);

// One lane of the block pipeline: a stream, its HBM buffers and the host-side scratch of one block.
// Blocks of a batch are decoded concurrently, one lane per host thread; the lanes' kernels and copies
// overlap on the device.
struct Lane {
  cudaStream_t st = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev_sync = nullptr;  // blocking-sync event: a waiting host thread sleeps instead of spinning
  ppd_stats stats{};
  DevBuf d_nodes, d_order, d_keys, d_vals, d_hashes, d_children, d_accounts, d_ref, d_ref_len, d_counters;
  DevBuf d_msg, d_msg_off, d_digest;
  DevBuf d_plan, d_out;  // IR dump plan and the serialised IrDump
  DevBuf d_wit, d_pa, d_pb, d_pc;  // witness bytes and the scratch of the three parse phases (ppd_parse.cu)
  DevBuf d_level, d_okeys, d_obins;  // node levels, and the scratch of the (level, class) ordering on the device
  DevBuf d_flat, d_txn, d_order2;    // the device txn loop (gpu_txn.cu): the resident FlatBlock, its tables and scratch, the order of its nodes
  cudaEvent_t ev_loop0 = nullptr, ev_loop1 = nullptr;
  uint32_t* h_parse = nullptr;     // page-locked landing area of the parse result words
  // the launch parameters of the lane's last GPU parse (the witness and all scratch stay resident), for ppd_replay_last_parse
  bool has_last_parse = false;
  ParseBounds last_bounds{};
  ParseEmit last_emit{};
  uint32_t* last_ins_pos = nullptr;
  uint32_t last_n_code = 0;
  size_t last_val_bytes = 0;
  Job* job = nullptr;  // page-locked pools, kept across calls
  // the arena of the lane's last block stays resident so that its hashing can be re-run for measurement
  bool has_last = false;
  ArenaView last_view{};
  std::vector<uint32_t> last_level_start, last_level_start2;  // (second sweep: the nodes the device txn loop appended, in d_order2)
  uint32_t last_n_msgs = 0;
  const uint8_t* last_msg_data = nullptr;  // null: the key messages are in d_msg / d_msg_off / d_digest
  const uint64_t* last_msg_se = nullptr;
  uint8_t* last_digest_out = nullptr;
  // the launch parameters of the lane's last device txn loop and IR dump, for ppd_replay_last_txn / ppd_replay_last_dump
  bool has_last_txn = false;
  txn::View last_txn{};
  txn::JoinView last_join{};
  txn::AcctInit last_ai{};
  txn::Cursors last_init{};
  uint32_t last_table_slots = 0, last_n_ops1 = 0, last_n_ops2 = 0, last_max_writes = 0, last_n_touched = 0, last_n_ir = 0, last_cap_tail = 0, last_max_keys = 0;
  uint32_t* last_bins_tail = nullptr;
  uint16_t* last_okeys = nullptr;
  IrDumpPlanView last_plan{};
  size_t last_out_bytes = 0;
  // PPD_TRACE: events recorded on the stream at stage boundaries, resolved into a timeline when the block is done
  std::vector<cudaEvent_t> tr_ev;
  std::vector<const char*> tr_label;
  std::vector<double> tr_host_ms;
  size_t tr_n = 0;
  int id = 0;
  CopyBatch copies;  // lane_copy: queued until lane_copy_flush (every wait flushes)
  // the stream pool (StreamPool below): `st` is the lane's own stream unless a decode holds one of the pool's
  cudaStream_t own_st = nullptr;
  struct StreamLease* lease = nullptr;
  txn::LoopTask* h_task = nullptr;  // page-locked: the kernel argument of a loop launched on the lane's own stream
  cudaEvent_t ev_ready = nullptr, ev_loop_done = nullptr;  // (ev_loop_done: blocking-sync)
};

// Counting semaphore: how many lanes may have their witness upload + parse in flight at once.  All lanes of a
// batch start together; letting every one of them share the copy engine and the SMs makes all of them finish
// their parse late and at the same time, after which all host threads shape their tries at once with the GPU
// idle.  Admitting a few at a time staggers the lanes, so the parse, the host shaping and the IR dump of
// different blocks overlap.
struct Slots {
  std::mutex mu;
  std::condition_variable cv;
  int free_slots;
  explicit Slots(int n) : free_slots(n) {}
  void acquire() {
    std::unique_lock<std::mutex> g(mu);
    cv.wait(g, [&] { return free_slots > 0; });
    free_slots--;
  }
  void release() {
    {
      std::lock_guard<std::mutex> g(mu);
      free_slots++;
    }
    cv.notify_one();
  }
};
struct SlotGuard {
  Slots* s;
  explicit SlotGuard(Slots* s_, double* wait_ms = nullptr) : s(s_) {
    if (!s) return;
    const auto t0 = std::chrono::steady_clock::now();
    s->acquire();
    if (wait_ms) *wait_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  }
  void done() {
    if (s) s->release();
    s = nullptr;
  }
  ~SlotGuard() { done(); }
};
// Lanes admitted at once.  A sweep of 12, 16 and 32 (profiles/r02b_knobs.txt: 512 config-2 blocks per stream call)
// moved no further from 8 than two runs at 8 differ (578 and 617 blocks/s); 32 gave 623, not re-measured.
constexpr int PARSE_SLOTS = 8;

}  // namespace ppd

namespace ppd {
// The device runs at most CUDA_DEVICE_MAX_CONNECTIONS (32) streams side by side: more streams share hardware queues, and
// a kernel waits for everything queued before it on ITS queue, whatever the stream.  So the lanes (one per block in
// flight: HBM buffers, host scratch, a host thread) do not own the streams their work runs on:
//   * a block holds one of the pool's main streams while it has short kernels and copies to queue (parse, hashing
//     sweeps, IR dump), and gives it back while its txn loop runs;
//   * the txn loops, the only long kernels (one resident thread block for milliseconds), run on a few loop streams,
//     the loops that are due together as ONE launch (LoopBatcher, gpu_txn.cu).
// Main + loop streams stay below 32, so nothing short ever queues behind a loop; blocks in flight are not limited by
// the stream count.
struct StreamPool {
  std::mutex mu;
  std::condition_variable cv;
  std::vector<cudaStream_t> all, free_;
  cudaStream_t acquire(double* wait_ms) {
    const auto t0 = std::chrono::steady_clock::now();
    std::unique_lock<std::mutex> g(mu);
    cv.wait(g, [&] { return !free_.empty(); });
    cudaStream_t s = free_.back();
    free_.pop_back();
    if (wait_ms) *wait_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return s;
  }
  void release(cudaStream_t s) {
    {
      std::lock_guard<std::mutex> g(mu);
      free_.push_back(s);
    }
    cv.notify_one();
  }
};
// a decode's hold on a pool stream (no pool, in the host-only profiling build PPD_HOSTPROF: the lane keeps its own stream)
struct StreamLease {
  StreamPool* pool;
  Lane* L;
  bool held = false;
  StreamLease(StreamPool* p, Lane* l) : pool(p), L(l) {
    L->lease = this;
    acquire();
  }
  void acquire() {
    if (!pool || held) return;
    L->st = pool->acquire(&L->stats.host_wait_ms);
    held = true;
  }
  void release() {  // (everything queued on it stays queued: streams are in order, the next holder's work runs behind it)
    if (!pool || !held) return;
    lane_copy_flush_fwd(L);
    pool->release(L->st);
    L->st = L->own_st;
    held = false;
  }
  ~StreamLease() {
    release();
    L->lease = nullptr;
  }
  static void lane_copy_flush_fwd(Lane* l);
};
struct LoopBatcher;
LoopBatcher* loop_batcher_create(int device, int n_streams);
void loop_batcher_destroy(LoopBatcher* b);
// queues the loop behind `ready` (an event recorded on the stream that prepared it), returns once it is launched; the
// caller then waits for `done`.  start / done: recorded on the loop stream around the launches.  Returns the launches.
uint32_t loop_batcher_run(LoopBatcher* b, const txn::View& v, uint32_t initial_state, uint32_t max_keys, cudaEvent_t ready, cudaEvent_t start,
                          cudaEvent_t done, cudaEvent_t done_blocking);
}  // namespace ppd

namespace ppd {
// The arrays of one trie the builder of ppd_build.cu made (BuildView): its structure, refs and branch bins.  A context
// owns one for its one-shot root and subset entries; a trie handle owns two (the current trie, and a spare that an
// update builds into).
struct BuildState {
  enum { B_L, B_M, B_LINKA, B_LINKB, B_BIDX, B_TMP, B_SMALL, B_DEPTH, B_REP, B_CHILD, B_ORDER, B_NCHILD, B_KEYS,
         B_REF, B_REF_LEN, B_IREF, B_IREF_LEN, B_COUNT };
  DevBuf d[B_COUNT];
  std::vector<uint32_t> end;  // host copy of the branch bins: depth 63 - g owns bins 16 g .. 16 g + 15 (end of each)
  uint32_t n = 0, nb = 0;     // leaves and branches of the trie last built
  void release() {
    for (DevBuf& b : d) b.release();
  }
};
}  // namespace ppd

struct ppd_ctx {
  int device = 0;
  ppd::StreamPool* pool = nullptr;      // (both null only in the host-only profiling build PPD_HOSTPROF)
  ppd::LoopBatcher* batcher = nullptr;
  ppd::Slots parse_slots_sem{ppd::PARSE_SLOTS};
  cudaStream_t st = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string err;
  std::mutex err_mu;
  ppd_stats stats{};
  std::vector<ppd::Lane*> lanes;
  size_t last_lanes_used = 0;  // lanes holding a resident block of the last decode call
  // HBM buffers of the non-block entry points, grown on demand and reused across calls
  ppd::DevBuf d_keys, d_vals, d_ref, d_ref_len, d_counters;
  ppd::DevBuf d_msg, d_msg_off, d_digest;
  ppd::BuildState build;     // the builder's arrays of the one-shot root and subset entries
  ppd::DevBuf d_leaves[24];  // sort / de-duplication / gather of ppd_trie_root_leaves[_dev], and an update's sort
  ppd::DevBuf d_subset[7];   // create_trie_subset of ppd_trie_subset_* (ppd_subset.cu), and an update's marking
  ppd::DevBuf d_merge[12];   // an update's merge and incremental hashing (ppd_update.cu)
  std::vector<ppd_trie*> tries;  // live trie handles (gpu_trie.cu), released with the context
};

namespace ppd {

void stats_reset(ppd_ctx* c);
void lane_sync(Lane* l);
// PPD_TRACE=<file>: one row per stage boundary of every block (lane, block, label, device ms, host ms since the
// context was made), for the pipeline timeline in profiles/.  Off: trace_mark costs one predictable branch.
// copy by kernel (CopyBatch): queue, and launch what is queued.  Anything launched after a flush sees the copies.
void lane_copy(Lane* l, void* dst, const void* src, size_t bytes);
void lane_copy_flush(Lane* l);
bool trace_on();
void trace_mark(Lane* l, const char* label);
void trace_flush(Lane* l);

// ============================================================================================
// Phase I: batched Keccak-256 of byte strings (addresses, slots, code)
// ============================================================================================
struct KeyHasher {
  PVec<uint8_t> data;
  std::vector<uint64_t> off{0};
  PVec<H256> digest;
  std::vector<uint64_t> lens;
  PVec<uint64_t> se;  // (begin, end) pairs
  KeyHasher() {
    data.alloc_fn = pinned_alloc, data.free_fn = pinned_free;
    digest.alloc_fn = pinned_alloc, digest.free_fn = pinned_free;
    se.alloc_fn = pinned_alloc, se.free_fn = pinned_free;
  }
  void reset() {
    data.clear(), digest.clear(), lens.clear(), se.clear();
    off.assign(1, 0);
  }
  uint32_t add(const uint8_t* p, size_t n) {
    size_t at = data.size(), padded = (n + 3) & ~(size_t)3;
    data.resize(at + padded);  // every message starts 4-byte aligned
    memcpy(data.data() + at, p, n);
    memset(data.data() + at + n, 0, padded - n);
    uint32_t idx = (uint32_t)lens.size();
    lens.push_back(n);
    off.push_back(data.size());
    return idx;
  }
  void run(Lane* c);  // ppd_host.cu
};

// ============================================================================================
// Compact witness -> instruction tree (compact_prestate_processing.rs:683-875, 387-668)
// ============================================================================================
struct Span {
  const uint8_t* p = nullptr;
  uint32_t n = 0;
};
// One instruction of the witness, 20 bytes.  Operands are not copied: `pos` points at the first operand
// byte and the (already validated) CBOR heads are re-read when the instruction is used.
struct WNode {
  uint32_t pos;
  uint8_t op, flags;     // flags: the account leaf's flag byte (bit0 code, bit1 storage, bit2 nonce, bit3 balance)
  uint16_t unused = 0;
  // tree links filled by the stack machine
  int32_t first_child;   // branch: first child (ascending nibble order); extension: child; account leaf: storage node
  int32_t next_sibling;  // next child of the same branch
  uint32_t aux;          // branch: the 32-bit mask; account leaf: code node (or ~0)
};

struct WCursor {
  const uint8_t* p;
  size_t n, pos = 0;
  uint8_t read_byte() {
    if (pos >= n) fail(PPD_ERR_UNEXPECTED_END_OF_STREAM, "read_byte at end of stream");
    return p[pos++];
  }
  bool cbor_head(uint8_t& major, uint64_t& arg) {
    if (pos >= n) return false;
    uint8_t b = p[pos++];
    major = b >> 5;
    uint8_t ai = b & 31;
    if (ai < 24) {
      arg = ai;
      return true;
    }
    if (ai > 27) return false;
    size_t w = (size_t)1 << (ai - 24);
    if (n - pos < w) return false;
    arg = 0;
    for (size_t i = 0; i < w; i++) arg = (arg << 8) | p[pos++];
    return true;
  }
  Span cbor_bytes(int err) {
    uint8_t major;
    uint64_t len;
    if (!cbor_head(major, len) || major != 2 || len > n - pos) fail(err, "bad CBOR byte string");
    Span s{p + pos, (uint32_t)len};
    pos += len;
    return s;
  }
  uint64_t cbor_uint(uint64_t max) {
    uint8_t major;
    uint64_t v;
    if (!cbor_head(major, v) || major != 0 || v > max) fail(PPD_ERR_INVALID_BYTES_FOR_TYPE, "bad CBOR unsigned integer");
    return v;
  }
};

// key_bytes_to_nibbles (compact_prestate_processing.rs:1338-1390); appends to `out`, returns count
inline uint32_t compact_key_nibbles(Span k, uint8_t* out) {
  if (k.n == 0) return 0;
  uint32_t c = 0;
  if (k.n == 1) {
    out[c++] = k.p[0] & 15;
    return c;
  }
  bool odd = k.p[0] & 1;
  uint32_t m = k.n - 1;
  if (2 * m > 64 + 1) fail(PPD_ERR_KEY_ERROR, "compact key longer than 64 nibbles");
  for (uint32_t i = 0; i + 1 < m; i++) {
    out[c++] = k.p[1 + i] >> 4;
    out[c++] = k.p[1 + i] & 15;
  }
  out[c++] = k.p[m] >> 4;
  if (!odd) out[c++] = k.p[m] & 15;
  return c;
}

// key_bytes_to_nibbles runs while the instructions are read (compact_prestate_processing.rs:787-835), so
// a key of more than 64 nibbles is reported in stream order, before any later parse error
inline void check_key_length(Span k) {
  if (k.n >= 2 && 2 * (k.n - 1) > 64 + 1) fail(PPD_ERR_KEY_ERROR, "compact key longer than 64 nibbles");
}

struct Witness {
  const uint8_t* bytes = nullptr;
  size_t len = 0;
  uint8_t version = 0;
  std::vector<WNode> ins;
  int32_t root = -1;  // -1: header only

  // operand views (the stream was validated by parse_witness)
  Span key(const WNode& x) const {
    WCursor c{bytes, len, x.pos};
    return c.cbor_bytes(PPD_ERR_INVALID_BYTE_VECTOR);
  }
  Span leaf_value(const WNode& x) const {
    WCursor c{bytes, len, x.pos};
    c.cbor_bytes(PPD_ERR_INVALID_BYTE_VECTOR);
    return c.cbor_bytes(PPD_ERR_INVALID_BYTE_VECTOR);
  }
  Span code(const WNode& x) const { return key(x); }
  const uint8_t* hash(const WNode& x) const { return bytes + x.pos; }
  void account(const WNode& x, Span& key_out, uint64_t& nonce, Span& balance) const {
    WCursor c{bytes, len, x.pos};
    key_out = c.cbor_bytes(PPD_ERR_INVALID_BYTE_VECTOR);
    c.pos++;  // flags
    nonce = (x.flags & 4) ? c.cbor_uint(~0ull) : 0;
    balance = (x.flags & 8) ? c.cbor_bytes(PPD_ERR_INVALID_BYTE_VECTOR) : Span{};
  }
};
void parse_witness(const uint8_t* w, size_t n, Witness& out);

struct TrieItem {
  uint32_t koff, klen;
  uint8_t kind;  // 0 value leaf, 1 account leaf, 2 hashed-out subtree
  uint32_t a1, a2;
};

// ============================================================================================
// One block being decoded
// ============================================================================================
struct TraceV {
  const uint8_t* addr;
  uint8_t flags;
  const uint8_t *balance = nullptr, *nonce = nullptr;
  uint32_t n_reads = 0, n_writes = 0;
  const uint8_t *reads = nullptr, *writes = nullptr;
  const uint8_t* code_read = nullptr;
  Span code_write;
  // message indices into the key hasher
  uint32_t m_addr = 0, m_reads = 0, m_writes_full = 0, m_writes_min = 0, m_code = 0;
};
struct TxnV {
  std::vector<TraceV> traces;
  Span byte_code, new_txn_node, new_receipt_node;
  uint64_t gas_used = 0;
};
struct FlatReader {
  const uint8_t* p;
  size_t n, pos = 0;
  void need(size_t k) {
    if (n - pos < k) fail(PPD_ERR_BAD_FLAT_INPUT, "flat block truncated");
  }
  uint8_t u8() {
    need(1);
    return p[pos++];
  }
  uint32_t u32() {
    need(4);
    uint32_t v;
    memcpy(&v, p + pos, 4);
    pos += 4;
    return v;
  }
  uint64_t u64() {
    need(8);
    uint64_t v;
    memcpy(&v, p + pos, 8);
    pos += 8;
    return v;
  }
  const uint8_t* raw(size_t k) {
    need(k);
    const uint8_t* r = p + pos;
    pos += k;
    return r;
  }
  Span bytes() {
    uint32_t k = u32();
    return Span{raw(k), k};
  }
};

struct IrPlan {
  uint64_t txn_before = 0, gas_before = 0, gas_after = 0;
  bool has_signed_txn = false;
  Span signed_txn;
  bool has_withdrawals = false;
  uint32_t state_sub = NODE_EMPTY, txn_sub = NODE_EMPTY, receipt_sub = NODE_EMPTY;  // roots of the tries the subsets are cut from
  std::vector<std::pair<H256, uint32_t>> storage_subs;
  std::vector<uint32_t> touched;
  uint32_t root_state = 0, root_txn = 0, root_receipt = 0;  // NK_ROOT nodes
  std::map<H256, Span> code;
};

struct BlockJob {
  // input views
  Span compact;
  uint32_t pre_image_kind = 0;         // 0 Combined{compact}; 2 Separate{Direct, MultipleTries{Direct}} (host_direct.cu)
  Span direct;                         // kind 2: the DirectPreImage payload; `compact` then points into Job::direct_wit
  std::vector<H256> direct_keep;       // kind 2: the hashed addresses that have a storage trie
  std::vector<TxnV> txns;
  std::unordered_map<H256, Span, H256Hasher> resolved_code;
  std::vector<std::pair<const uint8_t*, const uint8_t*>> withdrawals;
  std::vector<uint32_t> m_withdrawal_addr;
  const uint8_t* checkpoint = nullptr;
  Span b_meta, b_hashes;
  // decoded witness
  Witness wit;
  std::vector<uint32_t> m_inline_code;  // per instruction: message index of an inline Code node, or ~0
  std::map<H256, Span> pre_code;        // WitnessOutput.code
  // tries
  uint32_t state_root = NODE_EMPTY;
  H256Map storage;  // hashed address -> root node
  struct PreAccount {
    H256 haddr;
    uint32_t rec;
    bool storage_nonempty;
    bool witnesses_storage = false;  // its account leaf carries a storage node (flag bit 1)
    uint32_t own_root = NODE_EMPTY;  // root of the trie that node converts to
  };
  // a storage trie is witnessed only in part (it holds a hashed-out node): two accounts with the same storage root may
  // then be witnessed differently, and the reference's join by root hash (compact_to_partial_trie.rs:167-190) gives
  // both the trie witnessed last: resolved with the hashed roots before the txn loop (join_storage_by_root)
  bool storage_partial = false;
  bool pre_image_built = false;
  std::vector<PreAccount> pre_accounts;
  H256Map pre_with_storage;  // accounts whose storage root != EMPTY_TRIE_HASH -> record
  FlatMapU32 root_of;                                               // trie root node -> its NK_ROOT node
  std::unordered_map<int32_t, uint32_t> storage_root_of_instr;      // account leaf instruction -> root of its witnessed storage trie
  bool have_empty_form = false;                                     // a witnessed storage trie whose root is EMPTY_TRIE_HASH
  bool pre_image_on_gpu = false;                                    // gpu_pre_image built the pre-image tries
  uint32_t empty_form = NODE_EMPTY;
  std::vector<IrPlan> irs;
  int status = PPD_OK;
  std::string err;
};

void read_flat_block(const uint8_t* p, size_t n, BlockJob& b);
// host_direct.cu: a kind-2 pre-image as a compact witness written into `wit` (b.compact points there; b.direct_keep); the
// storage map cut to b.direct_keep
void direct_to_compact(BlockJob& b, PVec<uint8_t>& wit);
void direct_filter_storage(BlockJob& b);
// ---- minimal RLP helpers (structure only; no hashing): host_txn.cu ----
uint32_t u256_sig(const uint8_t* be);
void rlp_str(std::vector<uint8_t>& out, const uint8_t* p, size_t n);
void rlp_u256(std::vector<uint8_t>& out, const uint8_t* be);
struct RlpItem {
  bool is_list;
  const uint8_t* payload;
  size_t payload_len, total_len;
};
bool rlp_item(const uint8_t* p, size_t n, RlpItem& it);
bool is_legacy_receipt(const uint8_t* p, size_t n);

// ============================================================================================
// Job = a batch of blocks sharing one arena, one key-hash launch and one sweep
// ============================================================================================
struct Job {
  HostArena A;
  KeyHasher kh;
  std::vector<BlockJob> blocks;
  PVec<uint8_t> ref, ref_len;  // after the sweep
  PVec<uint32_t> order;
  PVec<uint32_t> plan;  // IR dump plan (inputs, then the outputs read back)
  PVec<uint8_t> out_stage;  // page-locked landing buffer of the serialised IrDump
  bool refs_on_host = false;
  // When the pre-image was built on the GPU (gpu_pre_image) the leading part of every pool is already in
  // the lane's device buffers: the sweep uploads only what the txn loop appended.  The value and hash
  // pools of that part are not copied to the host unless a host-side dump needs them (fetch_pools).
  struct Resident {
    size_t nodes = 0, keys = 0, vals = 0, hashes = 0, children = 0, accounts = 0;
  } dev;
  bool pools_on_host = true;
  PVec<uint32_t> acct_list, code_list;
  PVec<uint8_t> wit_stage;  // page-locked staging of a pageable witness
  // a kind-2 block's pre-image re-spelled as a witness (host_direct.cu), and the hashed addresses of its storage map
  // as the device's by-address join reads them: page-locked, read by the copy engine / copy kernel directly
  PVec<uint8_t> direct_wit;
  PVec<H256> direct_keep;
  std::vector<HostArena::MarkItem> mark_items;  // scratch of the txn loop
  std::vector<HostArena::BatchItem> batch_items;
  std::vector<uint32_t> haddr_keys, haddr_leaves;
  PVec<H256> code_digest;
  TxnTables txn;              // tables of the device txn loop (gpu_txn.cu)
  PVec<uint32_t> txn_host;    // page-locked landing area of its read-backs
  PVec<uint32_t> txn_export;  // ... and of the storage map a block with dummy entries reads back
  PVec<uint64_t> ir_base, big_off;
  PVec<uint32_t> big_cap;
  std::vector<uint32_t> stamp;
  uint32_t serial = 0;
  Job() {
    plan.alloc_fn = pinned_alloc, plan.free_fn = pinned_free;
    out_stage.alloc_fn = pinned_alloc, out_stage.free_fn = pinned_free;
    A.set_allocator(pinned_alloc, pinned_free);
    ref.alloc_fn = ref_len.alloc_fn = pinned_alloc, ref.free_fn = ref_len.free_fn = pinned_free;
    order.alloc_fn = pinned_alloc, order.free_fn = pinned_free;
    A.level.alloc_fn = pinned_alloc, A.level.free_fn = pinned_free;
    acct_list.alloc_fn = code_list.alloc_fn = pinned_alloc, acct_list.free_fn = code_list.free_fn = pinned_free;
    code_digest.alloc_fn = pinned_alloc, code_digest.free_fn = pinned_free;
    wit_stage.alloc_fn = pinned_alloc, wit_stage.free_fn = pinned_free;
    direct_wit.alloc_fn = direct_keep.alloc_fn = pinned_alloc, direct_wit.free_fn = direct_keep.free_fn = pinned_free;
    txn.set_allocator(pinned_alloc, pinned_free);
    txn_host.alloc_fn = pinned_alloc, txn_host.free_fn = pinned_free;
    txn_export.alloc_fn = pinned_alloc, txn_export.free_fn = pinned_free;
    ir_base.alloc_fn = pinned_alloc, ir_base.free_fn = pinned_free;
    big_off.alloc_fn = pinned_alloc, big_off.free_fn = pinned_free, big_cap.alloc_fn = pinned_alloc, big_cap.free_fn = pinned_free;
  }
  void reset(size_t n_blocks) {
    dev = Resident{};
    pools_on_host = true;
    A.clear();
    kh.reset();
    blocks.clear();
    blocks.resize(n_blocks);
    ref.clear(), ref_len.clear(), order.clear();
    serial = 0;
  }
};

Job& job_of(Lane* l, size_t n_blocks);
Lane* lane_of(ppd_ctx* c, size_t w);
void lane_delete(Lane* l);
void collect_witness_messages(Job& J, BlockJob& b);
void collect_messages(Job& J, BlockJob& b);
uint32_t root_node_for(Job& J, BlockJob& b, uint32_t trie_root);
void build_pre_image(Job& J, BlockJob& b);
void join_storage_by_root(Lane* L, Job& J, BlockJob& b);
bool gpu_parse_enabled();
// dev_only: the txn loop runs on the device too (gpu_txn.cu), so nothing of the arena is copied back: the witness is
// already resident (inside the uploaded FlatBlock), the pools get room for what the loop appends, and `after_launch`
// queues more work behind the emit kernels before the final wait
struct PreImageDeviceOnly {
  const uint8_t* d_witness;
  size_t extra_nodes, extra_children, extra_keys, extra_vals, extra_accounts;
  void (*after_launch)(void* arg, const ParseEmit& E);
  void* arg;
};
bool gpu_pre_image(Lane* L, Job& J, BlockJob& b, bool check_version = true, Slots* slots = nullptr, const PreImageDeviceOnly* dev_only = nullptr);
void upload_bytes(Lane* L, Job& J, uint8_t* dst, const uint8_t* src, size_t n);
void verify_gpu_pre_image(Lane* L, Job& J, BlockJob& b);
void shape_block(Job& J, BlockJob& b);
void sweep(Lane* c, Job& J, bool refs_to_host = true);
void fetch_refs(Lane* c, Job& J);
void fetch_pools(Lane* c, Job& J);

struct PhaseTimer {
  bool on = getenv("PPD_TIMING") != nullptr;
  std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
  void lap(const char* what) {
    if (!on) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[ppd] %-10s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t).count());
    t = now;
  }
};
// accumulating timer for the sections of the txn loop (PPD_TIMING only)
struct SectionTimer {
  bool on = getenv("PPD_TIMING") != nullptr;
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  std::chrono::steady_clock::time_point t;
  void start() {
    if (on) t = std::chrono::steady_clock::now();
  }
  void stop(int k) {
    if (!on) return;
    auto now = std::chrono::steady_clock::now();
    acc[k] += std::chrono::duration<double, std::milli>(now - t).count();
    t = now;
  }
  void report(const char* const* names, int n) {
    if (!on) return;
    for (int k = 0; k < n; k++) fprintf(stderr, "[ppd]   %-12s %8.3f ms\n", names[k], acc[k]);
  }
};

// ---- step 5: IrDump ------------------------------------------------------------------------------
// Growable byte buffer with unchecked-after-need() writes; give() hands the malloc'ed storage to the caller.
struct Out {
  uint8_t* p = nullptr;
  size_t n = 0, cap = 0;
  Out() {}
  Out(const Out&) = delete;
  Out& operator=(const Out&) = delete;
  Out(Out&& o) noexcept : p(o.p), n(o.n), cap(o.cap) { o.p = nullptr, o.n = o.cap = 0; }
  ~Out() { free(p); }
  void need(size_t k) {
    if (n + k <= cap) return;
    size_t nc = cap ? cap * 2 : 4096;
    while (nc < n + k) nc *= 2;
    uint8_t* q;
    if (nc >= (8u << 20)) {
      // large output buffers: 2 MiB-aligned and advised for transparent huge pages, so that first-touch
      // costs a few dozen page faults instead of thousands (free() releases it like any malloc block)
      nc = (nc + (2u << 20) - 1) & ~(size_t)((2u << 20) - 1);
      q = (uint8_t*)aligned_alloc(2u << 20, nc);
      if (q) {
        madvise(q, nc, MADV_HUGEPAGE);
        if (n) memcpy(q, p, n);
        free(p);
      }
    } else {
      q = (uint8_t*)realloc(p, nc);
    }
    if (!q) fail(PPD_ERR_BAD_ARGUMENT, "out of host memory");
    p = q, cap = nc;
  }
  void u8(uint8_t v) {
    need(1);
    p[n++] = v;
  }
  void u32(uint32_t v) {
    need(4);
    memcpy(p + n, &v, 4);
    n += 4;
  }
  void u64(uint64_t v) {
    need(8);
    memcpy(p + n, &v, 8);
    n += 8;
  }
  void raw(const uint8_t* q, size_t k) {
    need(k);
    if (k) memcpy(p + n, q, k);
    n += k;
  }
  void span(Span s) {
    u32(s.n);
    raw(s.p, s.n);
  }
  void u256(uint64_t v) {
    need(32);
    memset(p + n, 0, 24);
    for (int i = 0; i < 8; i++) p[n + 31 - i] = (uint8_t)(v >> (8 * i));
    n += 32;
  }
  uint8_t* give(size_t* len) {
    uint8_t* r = p ? p : (uint8_t*)malloc(1);
    *len = n;
    p = nullptr, n = cap = 0;
    return r;
  }
};

// per-thread marks of the nodes a subset keeps expanded
struct Stamp {
  std::vector<uint32_t> v;
  uint32_t serial = 0;
};

void dump_ir(const Job& J, const BlockJob& b, IrPlan& p, Stamp& st, Out& o);
void dump_blocks(Job& J, uint8_t** outs, size_t* out_lens, unsigned max_workers);
unsigned host_threads();

// Runs f(item, worker) for every item in [0, n) on up to `workers` threads (the caller's included).
template <class F>
void parallel_for(size_t n, unsigned workers, F f) {
  if (workers > n) workers = (unsigned)n;
  if (workers <= 1) {
    for (size_t i = 0; i < n; i++) f(i, 0u);
    return;
  }
  std::atomic<size_t> next{0};
  std::atomic<bool> failed{false};
  Fail first{PPD_OK, ""};
  std::mutex mu;
  auto body = [&](unsigned w) {
    for (;;) {
      size_t i = next.fetch_add(1);
      if (i >= n || failed.load()) return;
      try {
        f(i, w);
      } catch (const Fail& e) {
        std::lock_guard<std::mutex> g(mu);
        if (!failed.exchange(true)) first = e;
      } catch (const std::exception& e) {  // (an exception leaving a std::thread would terminate the process)
        std::lock_guard<std::mutex> g(mu);
        if (!failed.exchange(true)) first = Fail{PPD_ERR_BAD_ARGUMENT, e.what()};
      }
    }
  };
  std::vector<std::thread> th;
  for (unsigned w = 1; w < workers; w++) th.emplace_back(body, w);
  body(0);
  for (auto& t : th) t.join();
  if (failed.load()) throw first;
}

// ---- page-locked output buffers ---------------------------------------------------------------------
// The IrDump of a block is ~50 MB that the caller owns until ppd_free().  Handing out page-locked
// buffers from a process-wide pool lets the device write the result straight into the caller's buffer
// (no bounce copy, no first-touch page faults); ppd_free() returns the buffer to the pool.  The pool is
// capped (PPD_PINNED_OUT_MB, default 12288): beyond the cap outputs are ordinary malloc blocks.
struct OutPool {
  struct Entry {
    uint8_t* p;
    size_t cap;
    bool in_use;
  };
  std::mutex mu;
  std::vector<Entry> entries;
  size_t total = 0;
  size_t limit() {
    static size_t v = [] {
      const char* e = getenv("PPD_PINNED_OUT_MB");
      return (size_t)(e ? atoll(e) : 12288) << 20;
    }();
    return v;
  }
  uint8_t* take(size_t n) {
#ifdef PPD_HOSTPROF
    return nullptr;
#else
    std::lock_guard<std::mutex> g(mu);
    Entry* best = nullptr;
    for (Entry& e : entries)
      if (!e.in_use && e.cap >= n && (!best || e.cap < best->cap)) best = &e;
    if (best) {
      best->in_use = true;
      return best->p;
    }
    size_t cap = (n + (n >> 3) + (8u << 20) - 1) & ~(size_t)((8u << 20) - 1);
    if (total + cap > limit()) {
      // make room by releasing idle buffers that were too small
      for (size_t i = 0; i < entries.size() && total + cap > limit();)
        if (!entries[i].in_use) {
          cudaFreeHost(entries[i].p);
          total -= entries[i].cap;
          entries.erase(entries.begin() + i);
        } else {
          i++;
        }
      if (total + cap > limit()) return nullptr;
    }
    void* p = nullptr;
    if (cudaHostAlloc(&p, cap, cudaHostAllocPortable) != cudaSuccess) return nullptr;
    entries.push_back({(uint8_t*)p, cap, true});
    total += cap;
    return (uint8_t*)p;
#endif
  }
  bool give_back(void* p) {
    std::lock_guard<std::mutex> g(mu);
    for (Entry& e : entries)
      if (e.p == p) {
        e.in_use = false;
        return true;
      }
    return false;
  }
};
OutPool& out_pool();

bool gpu_txn_enabled();
enum { GPU_BLOCK_DECLINED = 0, GPU_BLOCK_DONE = 1 };
// the whole block on the device (gpu_txn.cu); DECLINED: nothing was produced, the host path decodes the block
int gpu_block(ppd_ctx* c, Lane* L, Job& J, const uint8_t* flat, size_t len, uint8_t** out, size_t* out_len);
bool gpu_dump_enabled();
enum { DUMP_ON_HOST = 0, DUMP_DONE = 1 };
int gpu_dump_block(ppd_ctx* c, Lane* L, Job& J, uint8_t** out, size_t* out_len);
void trie_release_all(ppd_ctx* c);  // ppd_ctx_destroy: every live trie handle (gpu_trie.cu)

// Runs an entry point's body: selects the context's device, and turns a Fail (or any exception) into a status code
// and the context's error message.
template <class F>
int guarded(ppd_ctx* c, F f) {
  if (!c) return PPD_ERR_BAD_ARGUMENT;
  try {
#ifndef PPD_HOSTPROF
    CUDA_OK(cudaSetDevice(c->device));
#endif
    f();
    return PPD_OK;
  } catch (const Fail& e) {
    c->err = e.msg;
    return e.code;
  } catch (const std::exception& e) {
    c->err = e.what();
    return PPD_ERR_BAD_ARGUMENT;
  }
}

}  // namespace ppd
