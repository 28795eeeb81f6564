// gpu_txn.cu — one block decoded with everything after the flat input on the device:
//
//   FlatBlock (host) ─H2D─► witness parse + pre-image arena        ppd_parse.cu   (gpu_pre_image, device-only mode)
//                         ► Keccak of addresses / slot keys / code  ppd_kernels.cu (ranges of the resident FlatBlock)
//                         ► pre-image hashed level by level         ppd_kernels.cu (the storage roots feed the by-root join)
//                         ► account join, op sort, THE TXN LOOP     ppd_txn.cu / txn_core.h
//                         ► the loop's new nodes hashed level by level
//                         ► every IR sized, laid out and written    ppd_dump.cu    ─D2H─► IrDump (host)
//
// The host reads the flat input, lays out descriptors and literals (txn_tables.cu) and launches; it shapes no trie,
// keeps no arena and copies nothing of the arena back.  Per block it waits five times for a few words (instruction
// count; pool sizes; code digests + level histogram; the loop's flag + cursors; IR sizes) and once for the output.
// A block the loop flags (an error the reference would report, or a capacity limit) is redone by the host path
// (decode_one in ppd_host.cu), which reports errors in the reference's order.
#include "host_pipeline.h"
#include "txn_tables.h"

namespace ppd {

bool gpu_txn_enabled() {
#ifdef PPD_HOSTPROF
  return false;
#else
  return gpu_parse_enabled() && gpu_dump_enabled() && getenv("PPD_HOST_TXN") == nullptr;  // read per call: the tests compare both paths
#endif
}

// ---- the txn loops of the blocks in flight, batched (host_pipeline.h: StreamPool) -------------------------------------
// A lane whose block is ready for its loop hands the task over and gives its main stream back; a service thread takes
// whatever tasks are waiting when a loop stream is free and launches them together, one thread block each.
struct LoopBatcher {
  static const int MAX_STREAMS = 16, BMAX = (int)LOOP_BATCH_MAX;
  struct Req {
    txn::LoopTask task;
    uint32_t n_txns = 0;
    cudaEvent_t ready = nullptr, start = nullptr, done = nullptr, done_blocking = nullptr;
    bool launched = false;
    uint32_t launches = 0;
    cudaError_t err = cudaSuccess;
  };
  struct LoopStream {
    cudaStream_t st = nullptr;
    cudaEvent_t idle = nullptr;     // recorded after a batch: the stream (and its task array) is free again when it has passed
    txn::LoopTask* tasks = nullptr;  // page-locked, BMAX entries: what the batch's launches read
  };
  int device = 0, n_streams = 0;
  LoopStream ls[MAX_STREAMS];
  std::mutex mu;
  std::condition_variable cv_work, cv_launched;
  std::deque<Req*> q;
  bool stop = false;
  std::thread th;

  void serve() {
#ifndef PPD_HOSTPROF
    cudaSetDevice(device);
    int next = 0;
    for (;;) {
      Req* batch[BMAX];
      int n = 0;
      {
        std::unique_lock<std::mutex> g(mu);
        cv_work.wait(g, [&] { return stop || !q.empty(); });
        if (stop && q.empty()) return;
      }
      // a free loop stream: the first whose last batch has ended, else wait for the one used longest ago
      int pick = -1;
      for (int k = 0; k < n_streams && pick < 0; k++) {
        const int s = (next + k) % n_streams;
        if (cudaEventQuery(ls[s].idle) == cudaSuccess) pick = s;
      }
      if (pick < 0) {
        pick = next;
        cudaEventSynchronize(ls[pick].idle);  // (tasks keep arriving meanwhile: they make the next batch)
      }
      next = (pick + 1) % n_streams;
      {
        std::lock_guard<std::mutex> g(mu);
        while (n < BMAX && !q.empty()) batch[n++] = q.front(), q.pop_front();
      }
      LoopStream& S = ls[pick];
      uint32_t max_txns = 0;
      bool any_shared = false;
      cudaError_t err = cudaSuccess;
      for (int k = 0; k < n; k++) {
        S.tasks[k] = batch[k]->task;
        max_txns = std::max(max_txns, batch[k]->n_txns);
        any_shared |= batch[k]->task.use_shared != 0;
        if (err == cudaSuccess) err = cudaStreamWaitEvent(S.st, batch[k]->ready, 0);
      }
      for (int k = 0; k < n && err == cudaSuccess; k++) err = cudaEventRecord(batch[k]->start, S.st);
      uint32_t launches = 0;
      if (err == cudaSuccess) {
        launches = launch_txn_loops(S.tasks, (uint32_t)n, max_txns, any_shared, S.st);
        err = cudaGetLastError();
      }
      for (int k = 0; k < n && err == cudaSuccess; k++) {
        err = cudaEventRecord(batch[k]->done, S.st);
        if (err == cudaSuccess) err = cudaEventRecord(batch[k]->done_blocking, S.st);
      }
      if (err == cudaSuccess) err = cudaEventRecord(S.idle, S.st);
      {
        std::lock_guard<std::mutex> g(mu);
        for (int k = 0; k < n; k++) batch[k]->launched = true, batch[k]->launches = launches, batch[k]->err = err;
      }
      cv_launched.notify_all();
    }
#endif
  }
};

LoopBatcher* loop_batcher_create(int device, int n_streams) {
#ifdef PPD_HOSTPROF
  return nullptr;
#else
  LoopBatcher* b = new LoopBatcher();
  b->device = device;
  b->n_streams = std::min(n_streams, (int)LoopBatcher::MAX_STREAMS);
  for (int k = 0; k < b->n_streams; k++) {
    LoopBatcher::LoopStream& S = b->ls[k];
    S.tasks = (txn::LoopTask*)pinned_alloc(sizeof(txn::LoopTask) * LoopBatcher::BMAX);
    if (!S.tasks || cudaStreamCreateWithFlags(&S.st, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&S.idle, cudaEventBlockingSync | cudaEventDisableTiming) != cudaSuccess || cudaEventRecord(S.idle, S.st) != cudaSuccess) {
      b->n_streams = k + 1;
      loop_batcher_destroy(b);
      return nullptr;
    }
  }
  b->th = std::thread([b] { b->serve(); });
  return b;
#endif
}
void loop_batcher_destroy(LoopBatcher* b) {
#ifndef PPD_HOSTPROF
  if (!b) return;
  if (b->th.joinable()) {
    {
      std::lock_guard<std::mutex> g(b->mu);
      b->stop = true;
    }
    b->cv_work.notify_all();
    b->th.join();
  }
  for (int k = 0; k < b->n_streams; k++) {
    if (b->ls[k].st) cudaStreamSynchronize(b->ls[k].st), cudaStreamDestroy(b->ls[k].st);
    if (b->ls[k].idle) cudaEventDestroy(b->ls[k].idle);
    if (b->ls[k].tasks) pinned_free(b->ls[k].tasks);
  }
  delete b;
#endif
}
uint32_t loop_batcher_run(LoopBatcher* b, const txn::View& v, uint32_t initial_state, uint32_t max_keys, cudaEvent_t ready, cudaEvent_t start,
                          cudaEvent_t done, cudaEvent_t done_blocking) {
#ifdef PPD_HOSTPROF
  return 0;
#else
  LoopBatcher::Req r;
  r.task.v = v, r.task.initial_state = initial_state, r.task.use_shared = txn_loop_uses_shared(max_keys);
  r.n_txns = v.n_txns, r.ready = ready, r.start = start, r.done = done, r.done_blocking = done_blocking;
  {
    std::lock_guard<std::mutex> g(b->mu);
    b->q.push_back(&r);
  }
  b->cv_work.notify_one();
  {
    std::unique_lock<std::mutex> g(b->mu);
    b->cv_launched.wait(g, [&] { return r.launched; });
  }
  CUDA_OK(r.err);
  return r.launches;
#endif
}

#ifndef PPD_HOSTPROF
namespace {

struct Carve2 {
  uint8_t* base;
  size_t off = 0;
  template <class T>
  T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* r = reinterpret_cast<T*>(base + off);
    off += count * sizeof(T);
    return r;
  }
};

// what the hook queued behind the emit kernels needs, and what it leaves for the rest of the pipeline
struct HookState {
  Lane* L;
  Job* J;
  TxnTables* T;
  const uint8_t* d_flat;
  size_t n_txns;
  const PVec<H256>* keep;  // a direct pre-image: the hashed addresses of its storage map (page-locked), else null
  // out
  TxnBases B{};
  txn::View v{};
  txn::JoinView j{};
  txn::AcctInit ai{};
  uint32_t table_slots = 0, n_pre_nodes = 0, cap_tail = 0;
  uint64_t* se = nullptr;
  uint32_t *bins_pre = nullptr, *bins_tail = nullptr;
  uint16_t* okeys = nullptr;
  txn::Withdrawal* d_withdrawals = nullptr;
  txn::AcctExport* d_export = nullptr;
  uint32_t* h_bins = nullptr;   // page-locked: [4096] pre-image bins, [4096] tail bins, then Cursors
  uint8_t* h_code_digests = nullptr;
};

void after_emit(void* arg, const ParseEmit& E) {
  HookState& H = *(HookState*)arg;
  Lane* L = H.L;
  Job& J = *H.J;
  TxnTables& T = *H.T;
  cudaStream_t st = L->st;
  const size_t n_nodes = J.dev.nodes, n_acct = J.dev.accounts, n_traces = T.traces.size();
  H.n_pre_nodes = (uint32_t)n_nodes;
  H.cap_tail = (uint32_t)T.est_nodes;
  // ---- where the loop's additions go in the pools ----
  TxnBases& B = H.B;
  B.dig_base = (uint32_t)((J.dev.keys + 31) & ~(size_t)31);
  B.txn_key_base = B.dig_base + 32u * T.n_msgs;
  B.key_cursor = B.txn_key_base + 12u * (uint32_t)H.n_txns;
  B.val_base = (uint32_t)((J.dev.vals + 3) & ~(size_t)3);
  B.rec_base = (uint32_t)n_acct;
  // ---- device memory of the loop ----
  uint32_t table = 64;
  while (table < 2 * n_traces) table <<= 1;
  const size_t n_keep = H.keep ? H.keep->size() : 0;
  uint32_t jtable = 64;
  while (jtable < 2 * std::max(n_acct, n_keep)) jtable <<= 1;
  H.table_slots = table;
  txn::View& v = H.v;
  txn::JoinView& j = H.j;
  const size_t n_sorted = std::max<size_t>(n_nodes, T.est_nodes);
  const size_t pc_slow_n = (size_t)T.max_ops * txn::PATH_CAP;  // (no txn has more path nodes than keys x path length)
  size_t pc_map_n = 64;
  while (pc_map_n < 2 * pc_slow_n) pc_map_n <<= 1;
  auto layout = [&](Carve2& c) {
    v.traces = c.take<txn::TxnTrace>(n_traces + 1);
    H.se = c.take<uint64_t>(2ull * T.n_msgs + 2);
    v.ops1 = c.take<txn::SOp>(T.n_ops1 + 1);
    v.ops2 = c.take<txn::SOp>(T.n_ops2 + 1);
    v.acct = c.take<txn::AcctState>(table);
    j.slot_owner = c.take<uint32_t>(jtable);
    j.slot_best = c.take<uint32_t>(jtable);
    j.join_storage = c.take<uint32_t>(n_acct + 1);
    j.join_root = c.take<uint32_t>(n_acct + 1);
    j.pre_flags = c.take<uint8_t>(n_acct + 1);
    j.keep = H.keep ? c.take<uint8_t>(32 * n_keep + 32) : nullptr;
    v.pre_slot = c.take<uint32_t>(n_acct + 1);
    H.d_withdrawals = c.take<txn::Withdrawal>(T.withdrawals.size() + 1);
    H.d_export = c.take<txn::AcctExport>(T.needs_dummies() ? n_acct + 1 : 1);
    v.s.path_node = c.take<uint32_t>((size_t)T.max_ops * txn::PATH_CAP + 1);
    v.s.path_pc = c.take<uint32_t>((size_t)T.max_ops * txn::PATH_CAP + 1);
    v.s.path_depth = c.take<uint8_t>((size_t)T.max_ops * txn::PATH_CAP + 1);
    v.s.plen = c.take<uint8_t>(T.max_ops + 1);
    v.s.tnode = c.take<uint32_t>(T.max_ops + 1);
    v.s.tpc = c.take<uint32_t>(T.max_ops + 1);
    v.s.tdepth = c.take<uint8_t>(T.max_ops + 1);
    v.s.tkind = c.take<uint8_t>(T.max_ops + 1);
    v.s.key_hi = c.take<uint32_t>(T.max_ops + 1);
    // the path-node table in HBM: everything for a txn whose keys do not fit in shared memory, the spill tier otherwise
    v.s.pc_slow = c.take<txn::PathNode>(pc_slow_n + 1);
    v.s.pc_map = c.take<uint32_t>(pc_map_n);
    v.s.pc_map_key = c.take<uint32_t>(pc_map_n);
    v.cur = c.take<txn::Cursors>(1);
    H.bins_pre = c.take<uint32_t>(ORDER_MAX_BINS);
    H.bins_tail = c.take<uint32_t>(ORDER_MAX_BINS);
    H.okeys = c.take<uint16_t>(n_sorted + 16);
  };
  {
    Carve2 sz{nullptr};
    layout(sz);
    L->d_txn.reserve(sz.off + 256);
    Carve2 c{L->d_txn.as<uint8_t>()};
    layout(c);
  }
  v.nodes = E.nodes, v.level = E.level, v.key_pool = E.key_pool, v.val_pool = E.val_pool, v.hash_pool = E.hash_pool;
  v.child_pool = E.child_pool, v.accounts = E.accounts;
  v.cap_nodes = (uint32_t)(n_nodes + T.est_nodes), v.cap_children = (uint32_t)(J.dev.children + T.est_children);
  v.cap_keys = (uint32_t)std::min<size_t>(L->d_keys.cap, 0xfffffff0u);
  v.flat = H.d_flat, v.n_txns = (uint32_t)H.n_txns, v.n_traces = (uint32_t)n_traces, v.dig_base = B.dig_base;
  v.rec_base = B.rec_base, v.val_base = B.val_base;
  v.pre_flags = j.pre_flags;
  v.s.pc_fast = nullptr, v.s.pc_n_fast = 0, v.s.pc_n_slow = (uint32_t)pc_slow_n, v.s.pc_map_mask = (uint32_t)pc_map_n - 1, v.s.pc_count = &v.cur->pc_count;
  v.s.sh_ops = nullptr;
  v.s.a_nodes = &v.cur->n_nodes, v.s.a_children = &v.cur->n_children, v.s.a_keys = &v.cur->key_bytes, v.s.a_max_level = &v.cur->max_level;
  v.withdrawals = H.d_withdrawals, v.n_withdrawals = (uint32_t)T.withdrawals.size();
  // (tables and read-backs go by kernel copy, lane_copy: the copy engines are left to the FlatBlock and the IrDump)
  lane_copy(L, H.d_withdrawals, T.withdrawals.data(), sizeof(txn::Withdrawal) * v.n_withdrawals);
  j.acct_list = E.acct_list, j.n_acct = (uint32_t)n_acct, j.table_mask = jtable - 1;
  if (H.keep) {
    j.n_keep = (uint32_t)n_keep;
    lane_copy(L, const_cast<uint8_t*>(j.keep), H.keep->data(), 32 * n_keep);
    L->stats.h2d_bytes += 32.0 * n_keep;
  }
  // ---- the byte strings to hash: straight out of the resident FlatBlock ----
  lane_copy(L, v.traces, T.traces.data(), sizeof(txn::TxnTrace) * n_traces);
  lane_copy_flush(L);
  L->stats.h2d_bytes += (double)(sizeof(txn::TxnTrace) * n_traces);
  launch_txn_msgs(v, H.se, st);
  launch_keccak256_ranges(H.d_flat, H.se, T.n_msgs, E.key_pool + B.dig_base, st);
  L->stats.kernel_launches += 2, L->stats.key_hashes += T.n_msgs;
  // the digests of written code are keys of the IRs' code maps, which the host sorts
  for (size_t k = 0; k < T.code_write_traces.size(); k++) {
    const uint32_t m = T.traces[T.code_write_traces[k]].m_code;
    lane_copy(L, H.h_code_digests + 32 * k, E.key_pool + B.dig_base + 32ull * m, 32);
  }
  // ---- pre-image nodes sorted by (level, class); the host needs where every level starts ----
  L->d_order.reserve(4ull * n_nodes + 16);
  CUDA_OK(cudaMemsetAsync(H.bins_pre, 0, 4ull * ORDER_MAX_BINS, st));
  launch_order_by_level_class(E.nodes, E.level, (uint32_t)n_nodes, ORDER_MAX_BINS, H.okeys, H.bins_pre, L->d_order.as<uint32_t>(), st);
  lane_copy(L, H.h_bins, H.bins_pre, 4ull * ORDER_MAX_BINS);
  L->stats.kernel_launches += 3, L->stats.d2h_bytes += 4.0 * ORDER_MAX_BINS;
}

// level_start[] from the bins the scatter left behind (bins[k] = end of bucket k; 64 buckets per level)
void levels_from_bins(const uint32_t* bins, uint32_t n, std::vector<uint32_t>& level_start) {
  level_start.assign(1, 0);
  for (uint32_t l = 0; l < ORDER_MAX_BINS / 64; l++) {
    const uint32_t end = bins[64 * l + 63];
    level_start.push_back(end);
    if (end >= n) break;
  }
}

}  // namespace
#endif

int gpu_block(ppd_ctx* c, Lane* L, Job& J, const uint8_t* flat, size_t len, uint8_t** out, size_t* out_len) {
#ifdef PPD_HOSTPROF
  return GPU_BLOCK_DECLINED;
#else
  BlockJob& b = J.blocks[0];
  if (!gpu_txn_enabled()) return GPU_BLOCK_DECLINED;
  {
    const char* e = getenv("PPD_GPU_PARSE_MIN_BYTES");
    const size_t min_bytes = e ? (size_t)atoll(e) : (size_t)512 << 10;
    if (b.compact.n < min_bytes || b.compact.n < 2) return GPU_BLOCK_DECLINED;
  }
  TxnTables& T = J.txn;
  PhaseTimer pt;
  if (!txn_tables_phase1(b, flat, len, T)) return GPU_BLOCK_DECLINED;
  pt.lap("t:tables1");
  cudaStream_t st = L->st;
  const ppd_stats stats0 = L->stats;
  // ---- the FlatBlock to the device; the witness inside it lands 256-byte aligned ----
  // A direct pre-image (kind 2) was re-spelled as a witness in the job's page-locked buffer: the witness gets a region of
  // its own after the FlatBlock, and of the FlatBlock only what follows the DirectPreImage payload goes up.  Nothing on
  // the device reads the payload or the header before it (every offset of the tables points past them), so the
  // pre-image crosses PCIe once.
  const bool direct = b.pre_image_kind == 2;
  const size_t up_from = direct ? (size_t)(b.direct.p - flat) + b.direct.n : 0;
  const size_t wit_off = direct ? (len + 256 + 255) & ~(size_t)255 : (size_t)(b.compact.p - flat);
  const size_t lead = direct ? 0 : (256 - (wit_off & 255)) & 255;
  L->d_flat.reserve(lead + (direct ? wit_off + b.compact.n + 256 : len + 512));
  uint8_t* d_flat = L->d_flat.as<uint8_t>() + lead;
  if (direct) {
    J.direct_keep.resize(b.direct_keep.size());
    if (!b.direct_keep.empty()) memcpy(J.direct_keep.data(), b.direct_keep.data(), sizeof(H256) * b.direct_keep.size());
  }
  L->tr_n = 0;
  trace_mark(L, "begin");
  upload_bytes(L, J, d_flat + up_from, flat + up_from, len - up_from);
  CUDA_OK(cudaMemsetAsync(d_flat + len, 0, 256, st));
  L->stats.h2d_bytes += (double)(len - up_from);
  if (direct) {
    // (page-locked: the copy engine reads it as it is; J.wit_stage may still feed the FlatBlock's copy)
    CUDA_OK(cudaMemcpyAsync(d_flat + wit_off, b.compact.p, b.compact.n, cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemsetAsync(d_flat + wit_off + b.compact.n, 0, 256, st));
    L->stats.h2d_bytes += (double)b.compact.n;
  }
  trace_mark(L, "uploaded");
  // page-locked landing areas
  const size_t h_words = 2 * ORDER_MAX_BINS + sizeof(txn::Cursors) / 4 + 64;
  J.txn_host.resize(h_words + 8 * T.code_write_traces.size() + 8);
  HookState H;
  H.L = L, H.J = &J, H.T = &T, H.d_flat = d_flat, H.n_txns = b.txns.size(), H.keep = direct ? &J.direct_keep : nullptr;
  H.h_bins = J.txn_host.data();
  H.h_code_digests = reinterpret_cast<uint8_t*>(J.txn_host.data() + h_words);
  PreImageDeviceOnly X{};
  X.d_witness = d_flat + wit_off;
  X.extra_nodes = T.est_nodes, X.extra_children = T.est_children;
  X.extra_keys = 64 + 32ull * T.n_msgs + 12ull * b.txns.size() + 40ull * (T.n_ops1 + T.n_ops2) + 4096;
  X.extra_vals = 64 + T.val_writes + 8ull * b.txns.size();
  for (const TxnV& tx : b.txns) X.extra_vals += tx.byte_code.n + tx.new_receipt_node.n;
  X.extra_accounts = T.n_recs + 1;
  X.after_launch = after_emit, X.arg = &H;
  if (!gpu_pre_image(L, J, b, true, &c->parse_slots_sem, &X)) {
    L->stats = stats0;
    return GPU_BLOCK_DECLINED;  // a witness the host builder takes (malformed, not canonical)
  }
  pt.lap("t:pre-image");
  trace_mark(L, "parsed");
  // ---- plan of every IR (needs the witness's code strings and the digests of written code) ----
  struct CD {
    HookState* H;
    TxnTables* T;
    std::vector<uint32_t> slot_of;  // trace -> index into h_code_digests
  } cd{&H, &T, {}};
  if (!T.code_write_traces.empty()) {
    cd.slot_of.assign(T.traces.size(), 0);
    for (size_t k = 0; k < T.code_write_traces.size(); k++) cd.slot_of[T.code_write_traces[k]] = (uint32_t)k;
  }
  auto code_digest = [](void* arg, uint32_t t) -> const uint8_t* {
    CD* x = (CD*)arg;
    return x->H->h_code_digests + 32ull * x->slot_of[t];
  };
  // (the plan copies code bytes out of the resident FlatBlock: a re-spelled witness has no code strings, so a direct
  // pre-image's code comes from the resolved-code table, which is inside it)
  if ((direct && !b.pre_code.empty()) || !txn_tables_phase2(b, flat, H.B, code_digest, &cd, T)) {
    L->stats = stats0;
    return GPU_BLOCK_DECLINED;
  }
  pt.lap("t:tables2");
  txn::View& v = H.v;
  const uint32_t n_ir = T.n_ir, n_seg = (uint32_t)T.seg_a.size(), n_touched = T.touched_begin[n_ir];
  const uint32_t n_pre = H.n_pre_nodes;
  // dummy entries list every storage trie of the state: their segments are appended after the loop (txn_tables_dummies)
  const int n_dummies = (T.dummy_initial[0] >= 0) + (T.dummy_initial[1] >= 0) + (T.dummy_final >= 0);
  const size_t dummy_entries = J.dev.accounts + T.traces.size();
  const size_t seg_cap = n_seg + (size_t)n_dummies * (2 * dummy_entries + 32), lit_cap = T.lit.size() + (size_t)n_dummies * (36 * dummy_entries + 512);
  // ---- the plan on the device: [txns | seg_a | seg_b | seg_c | seg_begin | touched_begin | lit | ir_base | touched |
  //                              seg_off | ir_size, ir_flag | ir_nuniq | u_node | u_size | u_off] ----
  // IRs whose touched list may hold more distinct nodes than a thread block's shared-memory set: their sets live in HBM
  PVec<uint64_t>& big_off = J.big_off;
  PVec<uint32_t>& big_cap = J.big_cap;
  big_off.resize(n_ir + 1), big_cap.resize(n_ir + 1);
  size_t big_words = 0;
  for (uint32_t i = 0; i < n_ir; i++) {
    const uint32_t tn = T.touched_begin[i + 1] - T.touched_begin[i];
    big_off[i] = ~0ull, big_cap[i] = 0;
    if (tn <= 2 * IR_SET_MAX_UNIQ) continue;
    uint32_t cap = 1u << 14;
    while (cap < 2 * tn) cap <<= 1;
    big_off[i] = big_words, big_cap[i] = cap;
    big_words += 3ull * cap;  // table keys, table slots, parents
  }
  IrDumpPlanView P{};
  uint64_t* d_big_off;
  uint32_t* d_big_cap;
  uint32_t *d_seg_a, *d_seg_b, *d_seg_c, *d_seg_begin, *d_seg_end, *d_touched_begin, *d_touched, *d_ir_size;
  uint64_t* d_ir_base;
  uint8_t* d_lit;
  txn::TxnDesc* d_txns;
  auto plan_layout = [&](Carve2& cv) {
    d_txns = cv.take<txn::TxnDesc>(n_ir + 1);
    d_seg_a = cv.take<uint32_t>(seg_cap + 1), d_seg_b = cv.take<uint32_t>(seg_cap + 1), d_seg_c = cv.take<uint32_t>(seg_cap + 1);
    d_seg_begin = cv.take<uint32_t>(n_ir + 1), d_seg_end = cv.take<uint32_t>(n_ir + 1), d_touched_begin = cv.take<uint32_t>(n_ir + 1);
    d_lit = cv.take<uint8_t>(lit_cap + 16);
    d_ir_base = cv.take<uint64_t>(n_ir + 1);
    d_touched = cv.take<uint32_t>((size_t)n_touched + 16);
    P.seg_off = cv.take<uint32_t>(seg_cap + 1);
    d_ir_size = cv.take<uint32_t>(2ull * n_ir + 2);  // ir_size, then ir_flag: read back together
    P.ir_nuniq = cv.take<uint32_t>(n_ir + 1);
    d_big_off = cv.take<uint64_t>(n_ir + 1), d_big_cap = cv.take<uint32_t>(n_ir + 1);
    P.big_scratch = cv.take<uint32_t>(big_words + 16);
    P.u_node = cv.take<uint32_t>((size_t)n_touched + 16), P.u_size = cv.take<uint32_t>((size_t)n_touched + 16), P.u_off = cv.take<uint32_t>((size_t)n_touched + 16);
  };
  {
    Carve2 sz{nullptr};
    plan_layout(sz);
    L->d_plan.reserve(sz.off + 256);
    Carve2 cv{L->d_plan.as<uint8_t>()};
    plan_layout(cv);
  }
  P.ir_size = d_ir_size, P.ir_flag = d_ir_size + n_ir;
  P.touched = d_touched, P.touched_begin = d_touched_begin, P.seg_a = d_seg_a, P.seg_b = d_seg_b, P.seg_c = d_seg_c, P.seg_begin = d_seg_begin;
  P.seg_end = d_seg_end;
  P.big_off = d_big_off, P.big_cap = d_big_cap;
  P.flat = d_flat, P.lit = d_lit, P.ir_base = d_ir_base;
  auto up = [&](void* dst, const void* src, size_t bytes) {
    if (!bytes) return;
    lane_copy(L, dst, src, bytes);
    L->stats.h2d_bytes += (double)bytes;
  };
  up(d_txns, T.txns.data(), sizeof(txn::TxnDesc) * T.txns.size());
  up(d_seg_a, T.seg_a.data(), 4ull * n_seg), up(d_seg_b, T.seg_b.data(), 4ull * n_seg), up(d_seg_c, T.seg_c.data(), 4ull * n_seg);
  up(d_touched_begin, T.touched_begin.data(), 4ull * (n_ir + 1));
  if (!n_dummies) up(d_seg_begin, T.seg_begin.data(), 4ull * (n_ir + 1)), up(d_seg_end, T.seg_end.data(), 4ull * (n_ir + 1));
  up(d_lit, T.lit.data(), T.lit.size());
  up(d_big_off, big_off.data(), 8ull * n_ir), up(d_big_cap, big_cap.data(), 4ull * n_ir);
  up(v.key_pool + H.B.txn_key_base, T.txn_keys.data(), T.txn_keys.size());
  lane_copy_flush(L);
  CUDA_OK(cudaMemsetAsync(d_touched, 0xff, 4ull * n_touched, st));
  v.txns = d_txns, v.touched = d_touched, v.seg_a = d_seg_a, v.seg_b = d_seg_b;
  // ---- the pre-image hashed: the storage roots decide which trie an account gets (the by-root join) ----
  std::vector<uint32_t> level_pre, level_tail;
  levels_from_bins(H.h_bins, n_pre, level_pre);
  L->d_ref.reserve(32ull * v.cap_nodes);
  L->d_ref_len.reserve(v.cap_nodes);
  L->d_counters.reserve(32);
  CUDA_OK(cudaMemsetAsync(L->d_counters.p, 0, 32, st));
  ArenaView V;
  V.nodes = v.nodes, V.key_pool = v.key_pool, V.val_pool = v.val_pool, V.hash_pool = v.hash_pool, V.child_pool = v.child_pool;
  V.accounts = v.accounts, V.ref = L->d_ref.as<uint8_t>(), V.ref_len = L->d_ref_len.as<uint8_t>();
  V.counters = L->d_counters.as<unsigned long long>();
  trace_mark(L, "plan_up");
  CUDA_OK(cudaEventRecord(L->ev0, st));
  for (size_t l = 0; l + 1 < level_pre.size(); l++) {
    launch_hash_level(V, L->d_order.as<uint32_t>(), level_pre[l], level_pre[l + 1], st);
    L->stats.kernel_launches++, L->stats.level_launches++;
  }
  CUDA_OK(cudaEventRecord(L->ev1, st));
  trace_mark(L, "pre_hashed");
  // ---- join (by root, or by address for a direct pre-image), account table, sorted ops, the loop ----
  H.j.ref = V.ref;
  CUDA_OK(cudaMemsetAsync(H.j.slot_owner, 0xff, 4ull * (H.j.table_mask + 1), st));
  CUDA_OK(cudaMemsetAsync(H.j.slot_best, 0, 4ull * (H.j.table_mask + 1), st));
  CUDA_OK(cudaMemsetAsync(v.pre_slot, 0xff, 4ull * (H.j.n_acct + 1), st));
  txn::Cursors init;
  memset(&init, 0, sizeof init);
  init.n_nodes = n_pre, init.n_children = (uint32_t)J.dev.children, init.key_bytes = H.B.key_cursor;
  init.state_root = b.state_root, init.txn_root = NODE_EMPTY, init.receipt_root = NODE_EMPTY;
  launch_txn_init(v, init, H.table_slots, st);
  H.j.flag = &v.cur->flag;
  if (direct)
    launch_join_by_address(v, H.j, st);
  else
    launch_join(H.j, st);
  H.ai = txn::AcctInit{H.table_slots - 1, b.state_root, H.j.join_storage, H.j.join_root};
  const uint32_t max_writes = T.max_trace_keys;
  L->stats.kernel_launches += 3 + launch_txn_prep(v, H.ai, T.n_ops1, T.n_ops2, max_writes, st);
#ifdef PPD_LOOP_PROF
  // development builds: the per-thread event log of one txn (PPD_LOOP_EVLOG=<txn>:<file>)
  static unsigned long long* d_evlog = nullptr;
  static uint32_t* d_evcount = nullptr;
  const uint32_t ev_cap = 1u << 16;
  const char* ev_env = getenv("PPD_LOOP_EVLOG");
  if (ev_env) {
    if (!d_evlog) {
      CUDA_OK(cudaMalloc(&d_evlog, 16ull * ev_cap));
      CUDA_OK(cudaMalloc(&d_evcount, 4));
    }
    CUDA_OK(cudaMemsetAsync(d_evcount, 0, 4, st));
    v.evlog = d_evlog, v.evcount = d_evcount, v.ev_txn = (uint32_t)atoi(ev_env), v.ev_cap = ev_cap;
  }
#endif
  trace_mark(L, "prep");
  // the loop runs on a loop stream, batched with the loops of other lanes that are due; this lane's main stream goes
  // back to the pool meanwhile
  lane_copy_flush(L);
  CUDA_OK(cudaEventRecord(L->ev_ready, st));
  L->lease->release();
  L->stats.kernel_launches += loop_batcher_run(c->batcher, v, b.state_root, T.max_ops, L->ev_ready, L->ev_loop0, L->ev_loop1, L->ev_loop_done);
  {
    const auto tw = std::chrono::steady_clock::now();
    CUDA_OK(cudaEventSynchronize(L->ev_loop_done));
    L->stats.host_wait_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tw).count();
  }
  L->lease->acquire();
  st = L->st;
  trace_mark(L, "loop");
  // ---- the loop's nodes sorted by (level, class) ----
  L->d_order2.reserve(4ull * H.cap_tail + 16);
  CUDA_OK(cudaMemsetAsync(H.bins_tail, 0, 4ull * ORDER_MAX_BINS, st));
  launch_order_by_level_class(v.nodes, v.level, H.cap_tail, ORDER_MAX_BINS, H.okeys, H.bins_tail, L->d_order2.as<uint32_t>(), st, n_pre, &v.cur->n_nodes);
  CUDA_OK(cudaGetLastError());
  txn::Cursors* h_cur = reinterpret_cast<txn::Cursors*>(H.h_bins + 2 * ORDER_MAX_BINS);
  lane_copy(L, H.h_bins + ORDER_MAX_BINS, H.bins_tail, 4ull * ORDER_MAX_BINS);
  lane_copy(L, h_cur, v.cur, sizeof(txn::Cursors));
  L->stats.kernel_launches += 3, L->stats.d2h_bytes += 4.0 * ORDER_MAX_BINS + sizeof(txn::Cursors);
  trace_mark(L, "tail_order");
  lane_sync(L);
  pt.lap("t:loop");
#ifdef PPD_LOOP_PROF
  if (ev_env && strchr(ev_env, ':')) {
    uint32_t n_ev = 0;
    CUDA_OK(cudaMemcpy(&n_ev, d_evcount, 4, cudaMemcpyDeviceToHost));
    n_ev = std::min(n_ev, ev_cap);
    std::vector<unsigned long long> ev(2ull * n_ev);
    if (n_ev) CUDA_OK(cudaMemcpy(ev.data(), d_evlog, 16ull * n_ev, cudaMemcpyDeviceToHost));
    if (FILE* f = fopen(strchr(ev_env, ':') + 1, "w")) {
      fprintf(f, "clock,thread,event\n");
      for (uint32_t k = 0; k < n_ev; k++) fprintf(f, "%llu,%llu,%llu\n", ev[2 * k], ev[2 * k + 1] >> 16, ev[2 * k + 1] & 0xffff);
      fclose(f);
    }
  }
#endif
  {
    float ms = 0;
    CUDA_OK(cudaEventElapsedTime(&ms, L->ev0, L->ev1));
    L->stats.gpu_ms += ms;
    CUDA_OK(cudaEventElapsedTime(&ms, L->ev_loop0, L->ev_loop1));
    L->stats.txn_gpu_ms += ms;
  }
  if (getenv("PPD_TIMING")) {
    const unsigned long long* pc = h_cur->phase_clocks;
    fprintf(stderr, "[ppd]   loop phases (Mclk): setup %.2f | walks %.2f | announce %.2f | storage tries up %.2f | records %.2f | state trie up %.2f | root nodes %.2f\n",
            pc[0] / 1e6, pc[1] / 1e6, pc[2] / 1e6, pc[3] / 1e6, pc[4] / 1e6, pc[5] / 1e6, pc[6] / 1e6);
  }
  if (h_cur->flag || h_cur->max_level >= ORDER_MAX_BINS / 64) {
    if (getenv("PPD_TIMING")) fprintf(stderr, "[ppd] device txn loop flag %u at txn %u (max level %u): host path\n", h_cur->flag, h_cur->flag_txn, h_cur->max_level);
    L->stats = stats0;
    L->has_last_parse = false;
    return GPU_BLOCK_DECLINED;
  }
  if (n_dummies) {
    // the storage map as it was before the first and is after the last txn, then the dummies' segments
    const size_t n_acct = J.dev.accounts, n_tr = T.traces.size();
    const size_t w_export = (sizeof(txn::AcctExport) * (n_acct + 1) + 3) / 4, w_table = (sizeof(txn::AcctState) * H.table_slots + 3) / 4, w_dig = 8 * (n_tr + 1);
    J.txn_export.resize(w_export + w_table + w_dig + 16);
    txn::AcctExport* h_export = reinterpret_cast<txn::AcctExport*>(J.txn_export.data());
    txn::AcctState* h_table = reinterpret_cast<txn::AcctState*>(J.txn_export.data() + w_export);
    uint8_t* h_dig = reinterpret_cast<uint8_t*>(J.txn_export.data() + w_export + w_table);
    launch_acct_export(v, H.j, H.d_export, st);
    CUDA_OK(cudaGetLastError());
    lane_copy(L, h_export, H.d_export, sizeof(txn::AcctExport) * n_acct);
    lane_copy(L, h_table, v.acct, sizeof(txn::AcctState) * H.table_slots);
    lane_copy(L, h_dig, v.key_pool + H.B.dig_base, 32ull * n_tr);
    L->stats.kernel_launches += 1, L->stats.d2h_bytes += (double)(sizeof(txn::AcctExport) * n_acct + sizeof(txn::AcctState) * H.table_slots + 32ull * n_tr);
    lane_sync(L);
    const size_t seg0 = T.seg_a.size(), lit0 = T.lit.size();
    txn_tables_dummies(b, flat, *h_cur, h_export, (uint32_t)n_acct, h_table, H.table_slots, h_dig, T);
    if (T.seg_a.size() > seg_cap || T.lit.size() > lit_cap) fail(PPD_ERR_BAD_ARGUMENT, "dummy entries exceed their plan space");
    up(d_seg_a + seg0, T.seg_a.data() + seg0, 4ull * (T.seg_a.size() - seg0)), up(d_seg_b + seg0, T.seg_b.data() + seg0, 4ull * (T.seg_b.size() - seg0));
    up(d_seg_c + seg0, T.seg_c.data() + seg0, 4ull * (T.seg_c.size() - seg0));
    up(d_lit + lit0, T.lit.data() + lit0, T.lit.size() - lit0);
    up(d_seg_begin, T.seg_begin.data(), 4ull * (n_ir + 1)), up(d_seg_end, T.seg_end.data(), 4ull * (n_ir + 1));
    lane_copy_flush(L);
    pt.lap("t:dummies");
  }
  const uint32_t n_total = h_cur->n_nodes, n_tail = n_total - n_pre;
  levels_from_bins(H.h_bins + ORDER_MAX_BINS, n_tail, level_tail);
  trace_mark(L, "host_resumed");
  CUDA_OK(cudaEventRecord(L->ev0, st));
  for (size_t l = 0; l + 1 < level_tail.size(); l++) {
    launch_hash_level(V, L->d_order2.as<uint32_t>(), level_tail[l], level_tail[l + 1], st);
    L->stats.kernel_launches++, L->stats.level_launches++;
  }
  CUDA_OK(cudaEventRecord(L->ev1, st));
  trace_mark(L, "tail_hashed");
  // ---- every IR sized and laid out ----
  CUDA_OK(cudaEventRecord(L->ev_loop0, st));
  launch_ir_size(V, P, n_ir, st);
  CUDA_OK(cudaEventRecord(L->ev_loop1, st));
  CUDA_OK(cudaGetLastError());
  J.plan.resize(2ull * n_ir + 8);
  uint32_t* h_sizes = J.plan.data();
  unsigned long long* h_counters = reinterpret_cast<unsigned long long*>(H.h_bins);  // (the pre-image bins are consumed)
  lane_copy(L, h_sizes, d_ir_size, 8ull * n_ir);
  lane_copy(L, h_counters, L->d_counters.p, 24);
  L->stats.kernel_launches += 1, L->stats.d2h_bytes += 8.0 * n_ir + 24;
  trace_mark(L, "ir_sized");
  lane_sync(L);
  pt.lap("t:sweep+size");
  {
    float ms = 0;
    CUDA_OK(cudaEventElapsedTime(&ms, L->ev0, L->ev1));
    L->stats.gpu_ms += ms;
    CUDA_OK(cudaEventElapsedTime(&ms, L->ev_loop0, L->ev_loop1));
    L->stats.dump_gpu_ms += ms;
  }
  L->stats.nodes_hashed += h_counters[0], L->stats.node_permutations += h_counters[1], L->stats.node_bytes += h_counters[2];
  L->stats.arena_nodes += n_total;
  L->stats.levels += level_pre.size() + level_tail.size() - 2;
  for (size_t m = 0; m < T.traces.size(); m++) {
    const txn::TxnTrace& tr = T.traces[m];
    L->stats.key_permutations += 1 + tr.n_reads + tr.n_writes + ((tr.flags & txn::TRF_MIN_KEYS) ? tr.n_writes : 0);
    if ((tr.flags & PPD_TR_CODE_WRITE) && !(tr.flags & PPD_TR_CODE_READ)) L->stats.key_permutations += tr.code_len / 136 + 1;
  }
  L->stats.marks_on_gpu += T.n_items;
  L->stats.txn_loops_on_gpu += 1;
  L->has_last = true, L->last_view = V;
  L->last_level_start = level_pre, L->last_level_start2 = level_tail, L->last_n_msgs = T.n_msgs;
  L->last_msg_data = d_flat, L->last_msg_se = H.se, L->last_digest_out = v.key_pool + H.B.dig_base;
  L->last_txn = H.v, L->last_join = H.j, L->last_ai = H.ai, L->last_init = init, L->last_table_slots = H.table_slots;
  L->last_n_ops1 = T.n_ops1, L->last_n_ops2 = T.n_ops2, L->last_max_writes = max_writes, L->last_n_touched = n_touched, L->last_max_keys = T.max_ops;
  L->last_plan = P, L->last_n_ir = n_ir, L->has_last_txn = true;
  L->last_cap_tail = H.cap_tail, L->last_bins_tail = H.bins_tail, L->last_okeys = H.okeys;
  // an IR the dump kernels cannot lay out (an untouched node shorter than 32 bytes that the subset keeps expanded, more
  // touched nodes than a thread block's set holds): the host path serialises such blocks
  uint64_t total = 8;
  PVec<uint64_t>& ir_base = J.ir_base;
  ir_base.resize(n_ir);
  for (uint32_t i = 0; i < n_ir; i++) {
    if (h_sizes[n_ir + i]) {
      if (getenv("PPD_TIMING")) fprintf(stderr, "[ppd] IR %u cannot be laid out on the device: host path\n", i);
      L->stats = stats0;
      L->has_last = L->has_last_parse = L->has_last_txn = false;
      return GPU_BLOCK_DECLINED;
    }
    ir_base[i] = total;
    total += h_sizes[i];
  }
  // ---- written on the device, copied back once ----
  Out o;
  uint8_t* pinned = total >= ((size_t)1 << 20) ? out_pool().take(total) : nullptr;
  if (!pinned) o.need(total);
  uint8_t* dst = pinned ? pinned : o.p;
  L->d_out.reserve(total + 64);
  L->last_out_bytes = total;
  up(d_ir_base, ir_base.data(), 8ull * n_ir);
  launch_store_u32x2(L->d_out.as<uint32_t>(), PPD_IR_DUMP_MAGIC, n_ir, st);
  L->stats.h2d_bytes += 8;
  lane_copy_flush(L);
  trace_mark(L, "host_resumed2");
  CUDA_OK(cudaEventRecord(L->ev0, st));
  launch_ir_emit(V, P, n_ir, L->d_out.as<uint8_t>(), st);
  CUDA_OK(cudaEventRecord(L->ev1, st));
  trace_mark(L, "ir_emitted");
  CUDA_OK(cudaGetLastError());
  L->stats.kernel_launches += 1;
  if (pinned) {
    const auto tw = std::chrono::steady_clock::now();
    cudaError_t e = cudaMemcpyAsync(dst, L->d_out.p, total, cudaMemcpyDeviceToHost, st);
    trace_mark(L, "downloaded");
    if (e == cudaSuccess) e = cudaEventRecord(L->ev_sync, st);
    if (e == cudaSuccess) e = cudaEventSynchronize(L->ev_sync);
    L->stats.host_wait_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tw).count();
    if (e != cudaSuccess) {
      out_pool().give_back(pinned);
      throw Fail{PPD_ERR_CUDA, std::string("IR dump copy: ") + cudaGetErrorString(e)};
    }
  } else {
    // pageable output: land the copy in the lane's page-locked buffer, then move it on
    J.out_stage.resize(total);
    CUDA_OK(cudaMemcpyAsync(J.out_stage.data(), L->d_out.p, total, cudaMemcpyDeviceToHost, st));
    lane_sync(L);
    memcpy(o.p, J.out_stage.data(), total);
    o.n = total;
  }
  L->stats.d2h_bytes += (double)total;
  {
    float ms = 0;
    CUDA_OK(cudaEventElapsedTime(&ms, L->ev0, L->ev1));
    L->stats.dump_gpu_ms += ms;
  }
  pt.lap("t:emit+copy");
  trace_mark(L, "end");
  trace_flush(L);
  if (pinned) {
    *out = pinned, *out_len = total;
  } else {
    *out = o.give(out_len);
  }
  return GPU_BLOCK_DONE;
#endif
}

}  // namespace ppd
