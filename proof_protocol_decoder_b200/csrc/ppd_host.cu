// ppd_host.cu — host side of libppd_b200.so: the C ABI (include/ppd_b200.h), the context that
// owns the stream and the HBM buffers, and the block pipeline
//
//   FlatBlock ─► parse witness (compact_prestate_processing.rs:683-875, 387-668)
//             ─► batch-hash every address / slot / code on the GPU      (utils.rs:11-13 call sites)
//             ─► shape all versions of all tries as one persistent DAG   (host_arena.h; no hashing)
//             ─► ONE level-synchronous GPU sweep over the DAG            (ppd_kernels.cu)
//             ─► serialise Vec<GenerationInputs> as an IrDump            (decoding.rs:131-145)
//
// The host never computes a Keccak or a node encoding.  If the CUDA device or the kernels are not
// usable every entry point fails with PPD_ERR_CUDA: there is no CPU fallback.
#include <time.h>

#include "host_pipeline.h"
#ifdef PPD_HOSTPROF
#include "../../tools/hostprof_stub.h"  // development-only host profiler build (tools/hostprof); never defined for libppd_b200.so
#endif

using namespace ppd;

namespace ppd {

#ifdef PPD_HOSTPROF
void* pinned_alloc(size_t n) { return malloc(n); }
void pinned_free(void* p) { free(p); }
#else
void* pinned_alloc(size_t n) {
  void* p = nullptr;
  return cudaHostAlloc(&p, n, cudaHostAllocDefault) == cudaSuccess ? p : nullptr;
}
void pinned_free(void* p) { cudaFreeHost(p); }
#endif

void stats_reset(ppd_ctx* c) { c->stats = ppd_stats{}; }

void StreamLease::lane_copy_flush_fwd(Lane* l) { lane_copy_flush(l); }
void lane_copy_flush(Lane* l) {
#ifndef PPD_HOSTPROF
  if (!l->copies.n) return;
  launch_copy_segments(l->copies, l->st);
  CUDA_OK(cudaGetLastError());
  l->stats.kernel_launches += 1;
  l->copies.n = 0;
#endif
}
void lane_copy(Lane* l, void* dst, const void* src, size_t bytes) {
  if (!bytes) return;
  if (l->copies.n == CopyBatch::MAX) lane_copy_flush(l);
  CopyBatch& b = l->copies;
  b.dst[b.n] = dst, b.src[b.n] = src, b.bytes[b.n] = bytes, b.n++;
}

// wait for everything queued on the lane's stream without spinning (lanes may outnumber cores)
void lane_sync(Lane* l) {
  lane_copy_flush(l);
  const auto t0 = std::chrono::steady_clock::now();
  CUDA_OK(cudaEventRecord(l->ev_sync, l->st));
  CUDA_OK(cudaEventSynchronize(l->ev_sync));
  l->stats.host_wait_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

// ---- PPD_TRACE ----
namespace {
struct TraceState {
  FILE* f = nullptr;
  cudaEvent_t base = nullptr;
  std::chrono::steady_clock::time_point host0;
  std::mutex mu;
  unsigned seq = 0;
};
TraceState& trace_state() {
  static TraceState* t = [] {
    TraceState* s = new TraceState;
#ifndef PPD_HOSTPROF
    const char* path = getenv("PPD_TRACE");
    if (path && *path && (s->f = fopen(path, "w")) != nullptr) {
      if (cudaEventCreate(&s->base) != cudaSuccess || cudaEventRecord(s->base, 0) != cudaSuccess || cudaEventSynchronize(s->base) != cudaSuccess) {
        fclose(s->f);
        s->f = nullptr;
      }
      s->host0 = std::chrono::steady_clock::now();
      if (s->f) fprintf(s->f, "lane,block,label,device_ms,host_ms\n");
    }
#endif
    return s;
  }();
  return *t;
}
}  // namespace
bool trace_on() { return trace_state().f != nullptr; }
void trace_mark(Lane* l, const char* label) {
#ifndef PPD_HOSTPROF
  TraceState& t = trace_state();
  if (!t.f) return;
  if (l->tr_n == l->tr_ev.size()) {
    cudaEvent_t e;
    CUDA_OK(cudaEventCreate(&e));
    l->tr_ev.push_back(e), l->tr_label.push_back(label), l->tr_host_ms.push_back(0);
  }
  CUDA_OK(cudaEventRecord(l->tr_ev[l->tr_n], l->st));
  l->tr_label[l->tr_n] = label;
  l->tr_host_ms[l->tr_n] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t.host0).count();
  l->tr_n++;
#endif
}
void trace_flush(Lane* l) {
#ifndef PPD_HOSTPROF
  TraceState& t = trace_state();
  if (!t.f || !l->tr_n) return;
  std::lock_guard<std::mutex> g(t.mu);
  const unsigned seq = t.seq++;
  for (size_t k = 0; k < l->tr_n; k++) {
    float ms = 0;
    if (cudaEventSynchronize(l->tr_ev[k]) != cudaSuccess || cudaEventElapsedTime(&ms, t.base, l->tr_ev[k]) != cudaSuccess) ms = -1;
    fprintf(t.f, "%d,%u,%s,%.4f,%.4f\n", l->id, seq, l->tr_label[k], ms, l->tr_host_ms[k]);
  }
  fflush(t.f);
  l->tr_n = 0;
#endif
}

void KeyHasher::run(Lane* c) {
  size_t n = lens.size();
  digest.resize(n);
  if (!n) return;
#ifdef PPD_HOSTPROF
  for (size_t i = 0; i < n; i++) hostprof::keccak256(data.data() + off[i], lens[i], digest[i].b);
  return;
#endif
  // messages are padded to 4-byte boundaries, so pass explicit (begin, end) pairs
  se.resize(2 * n);
  for (size_t i = 0; i < n; i++) se[2 * i] = off[i], se[2 * i + 1] = off[i] + lens[i];
  c->d_msg.reserve(data.size() + 16);
  c->d_msg_off.reserve(se.size() * 8);
  c->d_digest.reserve(n * 32);
  CUDA_OK(cudaMemcpyAsync(c->d_msg.p, data.data(), data.size(), cudaMemcpyHostToDevice, c->st));
  CUDA_OK(cudaMemcpyAsync(c->d_msg_off.p, se.data(), se.size() * 8, cudaMemcpyHostToDevice, c->st));
  launch_keccak256_ranges(c->d_msg.as<uint8_t>(), c->d_msg_off.as<uint64_t>(), (uint32_t)n, c->d_digest.as<uint8_t>(), c->st);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaMemcpyAsync(digest.data(), c->d_digest.p, n * 32, cudaMemcpyDeviceToHost, c->st));
  lane_sync(c);
  c->stats.key_hashes += n;
  for (size_t i = 0; i < n; i++) c->stats.key_permutations += lens[i] / 136 + 1;
  c->stats.h2d_bytes += (double)(data.size() + se.size() * 8);
  c->stats.d2h_bytes += (double)(n * 32);
  c->stats.kernel_launches += 1;
}

void job_delete(Job* j) { delete j; }
Job& job_of(Lane* l, size_t n_blocks) {
  if (!l->job) l->job = new Job();
  l->job->reset(n_blocks);
  return *l->job;
}

Lane* lane_of(ppd_ctx* c, size_t w) {
  while (c->lanes.size() <= w) {
    std::unique_ptr<Lane> l(new Lane());
    l->id = (int)c->lanes.size();
#ifndef PPD_HOSTPROF
    CUDA_OK(cudaStreamCreateWithFlags(&l->st, cudaStreamNonBlocking));
    l->own_st = l->st;
    l->h_task = (txn::LoopTask*)pinned_alloc(sizeof(txn::LoopTask));
    if (!l->h_task) fail(PPD_ERR_BAD_ARGUMENT, "out of page-locked memory");
    CUDA_OK(cudaEventCreateWithFlags(&l->ev_ready, cudaEventDisableTiming));
    CUDA_OK(cudaEventCreateWithFlags(&l->ev_loop_done, cudaEventBlockingSync | cudaEventDisableTiming));
    CUDA_OK(cudaEventCreate(&l->ev0));
    CUDA_OK(cudaEventCreate(&l->ev1));
    CUDA_OK(cudaEventCreateWithFlags(&l->ev_sync, cudaEventBlockingSync | cudaEventDisableTiming));
    CUDA_OK(cudaEventCreate(&l->ev_loop0));
    CUDA_OK(cudaEventCreate(&l->ev_loop1));
#endif
    c->lanes.push_back(l.release());
  }
  return c->lanes[w];
}
void lane_delete(Lane* l) {
#ifndef PPD_HOSTPROF
  DevBuf* bufs[] = {&l->d_nodes, &l->d_order,  &l->d_keys,     &l->d_vals, &l->d_hashes,  &l->d_children, &l->d_accounts,
                    &l->d_ref,   &l->d_ref_len, &l->d_counters, &l->d_msg,  &l->d_msg_off, &l->d_digest,
                    &l->d_plan,  &l->d_out,     &l->d_wit,      &l->d_pa,   &l->d_pb,      &l->d_pc,
                    &l->d_level, &l->d_okeys,   &l->d_obins,    &l->d_flat, &l->d_txn,     &l->d_order2};
  for (DevBuf* b : bufs) b->release();
  if (l->h_parse) pinned_free(l->h_parse);
  for (cudaEvent_t e : l->tr_ev) cudaEventDestroy(e);
  if (l->h_task) pinned_free(l->h_task);
  if (l->ev_ready) cudaEventDestroy(l->ev_ready);
  if (l->ev_loop_done) cudaEventDestroy(l->ev_loop_done);
  if (l->ev0) cudaEventDestroy(l->ev0);
  if (l->ev1) cudaEventDestroy(l->ev1);
  if (l->ev_sync) cudaEventDestroy(l->ev_sync);
  if (l->ev_loop0) cudaEventDestroy(l->ev_loop0);
  if (l->ev_loop1) cudaEventDestroy(l->ev_loop1);
  if (l->st) cudaStreamDestroy(l->st);
#endif
  if (l->job) job_delete(l->job);
  delete l;
}

// ---- step 4: the sweep ---------------------------------------------------------------------------
void sweep(Lane* c, Job& J, bool refs_to_host) {
  HostArena& A = J.A;
  uint32_t n = (uint32_t)A.nodes.size();
  J.ref.resize(32ull * n);
  J.ref_len.resize(n);
  J.refs_on_host = true;
  if (!n) return;
#ifdef PPD_HOSTPROF
  memset(J.ref.data(), 0, 32ull * n);
  memset(J.ref_len.data(), 32, n);
  return;
#endif
  // node ids counting-sorted by (level, class): inside a level, nodes of one kind and one permutation count are
  // adjacent, so the lanes of a warp do the same work.  The sort itself runs on the device (ppd_kernels.cu:
  // launch_order_by_level_class); the host only needs where every level starts.
  uint32_t n_levels = 0;
  for (uint32_t i = 0; i < n; i++) n_levels = std::max<uint32_t>(n_levels, A.level[i] + 1u);
  std::vector<uint32_t> level_start(n_levels + 1, 0);
  for (uint32_t i = 0; i < n; i++) level_start[A.level[i] + 1u]++;
  for (uint32_t l = 0; l < n_levels; l++) level_start[l + 1] += level_start[l];
  const bool device_order = 64u * n_levels <= ORDER_MAX_BINS;
  PVec<uint32_t>& order = J.order;
  if (!device_order) {  // a trie deeper than 64 levels: the same sort on the host
    auto node_class = [&](uint32_t i) -> uint32_t {
      const NodeRec& r = A.nodes[i];
      uint32_t kind = r.w0 & 0xff;
      if (kind == NK_BRANCH) return 40 + ((uint32_t)__builtin_popcount(r.a1 & 0xffff) - 1 & 15);  // by child count
      if (kind == NK_ROOT) return 56;
      uint32_t perms = 1;
      if (kind == NK_LEAF) {
        uint32_t nl = (r.w0 >> 16) & 0xff;
        perms = ((nl < 2 ? 1 : 2 + (nl >> 1)) + r.a2 + 6) / 136 + 1;  // header bytes over-estimated by at most 3
      }
      return kind * 8 + (perms > 8 ? 7 : perms - 1);
    };
    order.resize(n);
    std::vector<uint8_t> cls(n);
    std::vector<uint32_t> bucket((size_t)n_levels * 64 + 1, 0);
    for (uint32_t i = 0; i < n; i++) {
      cls[i] = (uint8_t)node_class(i);
      bucket[(size_t)A.level[i] * 64 + cls[i] + 1]++;
    }
    for (size_t k = 0; k + 1 < bucket.size(); k++) bucket[k + 1] += bucket[k];
    for (uint32_t i = 0; i < n; i++) order[bucket[(size_t)A.level[i] * 64 + cls[i]]++] = i;
  }
  // the part of every pool that gpu_pre_image left in the lane's buffers stays where it is
  const Job::Resident& R = J.dev;
  c->d_nodes.reserve_keep(16ull * n, 16ull * R.nodes, c->st);
  c->d_order.reserve(4ull * n);
  c->d_keys.reserve_keep(A.key_pool.size() + 16, R.keys, c->st);
  c->d_vals.reserve_keep(A.val_pool.size() + 16, R.vals, c->st);
  c->d_hashes.reserve_keep(A.hash_pool.size() + 32, R.hashes, c->st);
  c->d_children.reserve_keep(4ull * A.child_pool.size() + 16, 4ull * R.children, c->st);
  c->d_accounts.reserve_keep(sizeof(AccountRec) * A.accounts.size() + 16, sizeof(AccountRec) * R.accounts, c->st);
  c->d_ref.reserve(32ull * n);
  c->d_ref_len.reserve(n);
  c->d_counters.reserve(32);
  auto up = [&](DevBuf& d, const void* src, size_t bytes, size_t resident = 0) {
    if (bytes <= resident) return;
    CUDA_OK(cudaMemcpyAsync(d.as<uint8_t>() + resident, (const uint8_t*)src + resident, bytes - resident, cudaMemcpyHostToDevice, c->st));
    c->stats.h2d_bytes += (double)(bytes - resident);
  };
  up(c->d_nodes, A.nodes.data(), 16ull * n, 16ull * R.nodes);
  if (device_order) {
    c->d_level.reserve_keep(2ull * n + 16, 2ull * R.nodes, c->st);
    c->d_okeys.reserve(2ull * n + 16);
    c->d_obins.reserve(4ull * ORDER_MAX_BINS);
    up(c->d_level, A.level.data(), 2ull * n, 2ull * R.nodes);
    CUDA_OK(cudaMemsetAsync(c->d_obins.p, 0, 4ull * 64 * n_levels, c->st));
    launch_order_by_level_class(c->d_nodes.as<NodeRec>(), c->d_level.as<uint16_t>(), n, 64 * n_levels, c->d_okeys.as<uint16_t>(),
                                c->d_obins.as<uint32_t>(), c->d_order.as<uint32_t>(), c->st);
    c->stats.kernel_launches += 3;
  } else {
    up(c->d_order, order.data(), 4ull * n);
  }
  up(c->d_keys, A.key_pool.data(), A.key_pool.size(), R.keys);
  up(c->d_vals, A.val_pool.data(), A.val_pool.size(), R.vals);
  up(c->d_hashes, A.hash_pool.data(), A.hash_pool.size(), R.hashes);
  up(c->d_children, A.child_pool.data(), 4ull * A.child_pool.size(), 4ull * R.children);
  up(c->d_accounts, A.accounts.data(), sizeof(AccountRec) * A.accounts.size(), sizeof(AccountRec) * R.accounts);
  CUDA_OK(cudaMemsetAsync(c->d_counters.p, 0, 32, c->st));
  ArenaView V;
  V.nodes = c->d_nodes.as<NodeRec>();
  V.key_pool = c->d_keys.as<uint8_t>();
  V.val_pool = c->d_vals.as<uint8_t>();
  V.hash_pool = c->d_hashes.as<uint8_t>();
  V.child_pool = c->d_children.as<uint32_t>();
  V.accounts = c->d_accounts.as<AccountRec>();
  V.ref = c->d_ref.as<uint8_t>();
  V.ref_len = c->d_ref_len.as<uint8_t>();
  V.counters = c->d_counters.as<unsigned long long>();
  CUDA_OK(cudaEventRecord(c->ev0, c->st));
  for (uint32_t l = 0; l < n_levels; l++) {
    launch_hash_level(V, c->d_order.as<uint32_t>(), level_start[l], level_start[l + 1], c->st);
    c->stats.kernel_launches++;
    c->stats.level_launches++;
  }
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaEventRecord(c->ev1, c->st));
  unsigned long long counters[3] = {0, 0, 0};
  c->has_last = true;
  c->last_view = V;
  c->last_level_start = level_start;
  c->last_level_start2.clear();
  c->last_msg_data = nullptr;
  c->has_last_txn = false;
  c->last_n_msgs = (uint32_t)J.kh.lens.size();
  J.refs_on_host = refs_to_host;
  if (refs_to_host) {
    CUDA_OK(cudaMemcpyAsync(J.ref.data(), c->d_ref.p, 32ull * n, cudaMemcpyDeviceToHost, c->st));
    CUDA_OK(cudaMemcpyAsync(J.ref_len.data(), c->d_ref_len.p, n, cudaMemcpyDeviceToHost, c->st));
  }
  CUDA_OK(cudaMemcpyAsync(counters, c->d_counters.p, 24, cudaMemcpyDeviceToHost, c->st));
  lane_sync(c);
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  c->stats.gpu_ms += ms;
  c->stats.nodes_hashed += counters[0];
  c->stats.node_permutations += counters[1];
  c->stats.node_bytes += counters[2];
  c->stats.arena_nodes += n;
  c->stats.levels += n_levels;
  if (refs_to_host) c->stats.d2h_bytes += 33.0 * n;
}

// the refs of the last sweep, for the host paths that need them (host IR serialisation)
void fetch_refs(Lane* c, Job& J) {
  if (J.refs_on_host) return;
  size_t n = J.A.nodes.size();
  CUDA_OK(cudaMemcpyAsync(J.ref.data(), c->d_ref.p, 32ull * n, cudaMemcpyDeviceToHost, c->st));
  CUDA_OK(cudaMemcpyAsync(J.ref_len.data(), c->d_ref_len.p, n, cudaMemcpyDeviceToHost, c->st));
  lane_sync(c);
  c->stats.d2h_bytes += 33.0 * n;
  J.refs_on_host = true;
}

// the value and hash pools of a GPU-built pre-image, for the host paths that read them (host IR serialisation)
void fetch_pools(Lane* c, Job& J) {
  if (J.pools_on_host) return;
  if (J.dev.vals) CUDA_OK(cudaMemcpyAsync(J.A.val_pool.data(), c->d_vals.p, J.dev.vals, cudaMemcpyDeviceToHost, c->st));
  if (J.dev.hashes) CUDA_OK(cudaMemcpyAsync(J.A.hash_pool.data(), c->d_hashes.p, J.dev.hashes, cudaMemcpyDeviceToHost, c->st));
  lane_sync(c);
  c->stats.d2h_bytes += (double)(J.dev.vals + J.dev.hashes);
  J.pools_on_host = true;
}

}  // namespace ppd


namespace ppd {
OutPool& out_pool() {
  static OutPool* p = new OutPool();  // never destroyed: buffers may outlive every context
  return *p;
}
}  // namespace ppd

namespace {

// One block on one lane: parse, key hashes, shaping, sweep, dump.  A failure that is the block's own
// (bad input, a reference panic site) is reported through *status; a CUDA failure is thrown.
void decode_one_inner(ppd_ctx* c, Lane* L, const uint8_t* flat, size_t len, uint8_t** out, size_t* out_len, int* status, unsigned dump_workers);
// host_busy_ms: the CPU time the block cost its host thread (CLOCK_THREAD_CPUTIME_ID: sleeping for the device or for a
// stream does not count, polling does) — the quantity that bounds blocks/s when several GPUs share the host's cores
static double thread_cpu_ms() {
  timespec ts;
  clock_gettime(CLOCK_THREAD_CPUTIME_ID, &ts);
  return 1e3 * (double)ts.tv_sec + 1e-6 * (double)ts.tv_nsec;
}
void decode_one(ppd_ctx* c, Lane* L, const uint8_t* flat, size_t len, uint8_t** out, size_t* out_len, int* status, unsigned dump_workers) {
  const double t0 = thread_cpu_ms();
  decode_one_inner(c, L, flat, len, out, out_len, status, dump_workers);
  L->stats.host_busy_ms += thread_cpu_ms() - t0;
}
void decode_one_inner(ppd_ctx* c, Lane* L, const uint8_t* flat, size_t len, uint8_t** out, size_t* out_len, int* status, unsigned dump_workers) {
  *out = nullptr, *out_len = 0;
  // First everything after the flat input on the device (gpu_txn.cu).  A block it declines (an error the reference
  // would report, a witness the GPU parser hands to the host builder, a capacity limit) starts over on the host path:
  // the host shapes the tries, in the reference's order of operations, and the device hashes and serialises them.
  StreamLease lease(c->pool, L);
  // a direct pre-image (kind 2) is re-spelled as a witness once, into the job's page-locked buffer; a block the device
  // declines keeps it (and its map's addresses) for the host attempt
  Span respelled{};
  std::vector<H256> keep;
  for (int on_device = gpu_txn_enabled() ? 1 : 0; on_device >= 0; on_device--) {
    PhaseTimer pt;
    Job& J = job_of(L, 1);
    BlockJob& b = J.blocks[0];
    try {
      read_flat_block(flat, len, b);
      pt.lap("read-flat");
      if (b.pre_image_kind == 2) {
        if (!respelled.p) {
          direct_to_compact(b, J.direct_wit);
          pt.lap("direct");
        } else {
          b.compact = respelled, b.direct_keep.swap(keep);
        }
      }
      if (on_device) {
        if (gpu_block(c, L, J, flat, len, out, out_len) == GPU_BLOCK_DONE) {
          *status = PPD_OK;
          return;
        }
        if (b.pre_image_kind == 2) respelled = b.compact, keep.swap(b.direct_keep);
        continue;
      }
      if (gpu_parse_enabled()) gpu_pre_image(L, J, b, true, &c->parse_slots_sem);
      collect_messages(J, b);
      pt.lap("parse");
      J.kh.run(L);
      pt.lap("keyhash");
      if (!b.pre_image_built) build_pre_image(J, b);
      if (b.pre_image_kind == 2)
        direct_filter_storage(b);
      else if (b.storage_partial)
        join_storage_by_root(L, J, b);
      shape_block(J, b);
      pt.lap("shape");
      sweep(L, J, /*refs_to_host=*/!gpu_dump_enabled());
      pt.lap("sweep");
      if (gpu_dump_block(c, L, J, out, out_len) == DUMP_ON_HOST) {
        fetch_refs(L, J);
        fetch_pools(L, J);
        dump_blocks(J, out, out_len, dump_workers);
      }
      pt.lap("dump");
      *status = PPD_OK;
      return;
    } catch (const std::bad_alloc&) {
      *status = PPD_ERR_BAD_FLAT_INPUT;  // sizes taken from the input that no memory can hold
      std::lock_guard<std::mutex> g(c->err_mu);
      c->err = "out of memory while reading the block";
      return;
    } catch (const Fail& e) {
      if (e.code == PPD_ERR_CUDA) throw;
      *status = e.code;
      std::lock_guard<std::mutex> g(c->err_mu);
      c->err = e.msg;
      return;
    }
  }
}

void add_stats(ppd_stats& a, const ppd_stats& b) {
  a.nodes_hashed += b.nodes_hashed, a.node_permutations += b.node_permutations, a.key_hashes += b.key_hashes;
  a.key_permutations += b.key_permutations, a.node_bytes += b.node_bytes, a.arena_nodes += b.arena_nodes;
  a.levels = std::max(a.levels, b.levels);
  a.gpu_ms += b.gpu_ms, a.h2d_bytes += b.h2d_bytes, a.d2h_bytes += b.d2h_bytes, a.kernel_launches += b.kernel_launches;
  a.witnesses_on_gpu += b.witnesses_on_gpu, a.witness_instructions += b.witness_instructions, a.witness_bytes += b.witness_bytes;
  a.parse_gpu_ms += b.parse_gpu_ms, a.level_launches += b.level_launches, a.marks_on_gpu += b.marks_on_gpu;
  a.txn_loops_on_gpu += b.txn_loops_on_gpu, a.txn_gpu_ms += b.txn_gpu_ms, a.dump_gpu_ms += b.dump_gpu_ms;
  a.host_busy_ms += b.host_busy_ms, a.host_wait_ms += b.host_wait_ms;
}

// Blocks are independent (each BlockTrace carries its own pre-image, trace_protocol.rs:40-48): every
// host thread takes blocks on its own lane, so parsing / shaping of one block overlaps the copies and
// kernels of the others.
static const size_t MAX_LANES = 64, LANES_CAP = 128;
static size_t max_lanes() {
  static const size_t n = [] {
    const char* e = getenv("PPD_MAX_LANES");
    const long v = e ? atol(e) : (long)MAX_LANES;
    return (size_t)(v < 1 ? 1 : v > (long)LANES_CAP ? (long)LANES_CAP : v);
  }();
  return n;
}

void decode_blocks(ppd_ctx* c, const uint8_t* const* flats, const size_t* lens, size_t n, uint8_t** outs, size_t* out_lens, int* statuses,
                   ppd_block_done_fn done = nullptr, void* user = nullptr) {
  stats_reset(c);
  if (!n) return;
  // block i runs on lane i mod n_lanes; a host thread takes whole lanes, so a lane never runs two
  // blocks at once and the last block of every lane stays resident in HBM (ppd_replay_last_hashing)
  const size_t n_lanes = std::min(n, max_lanes());
  const unsigned workers = (unsigned)std::min<size_t>(host_threads(), n_lanes);
  for (size_t w = 0; w < n_lanes; w++) {
    Lane* L = lane_of(c, w);
    L->stats = ppd_stats{};
    L->has_last = false;
    L->has_last_parse = false;
    L->has_last_txn = false;
  }
  const unsigned dump_workers = std::max(1u, host_threads() / workers);
  for (size_t i = 0; i < n; i++) outs[i] = nullptr, out_lens[i] = 0, statuses[i] = PPD_OK;
  parallel_for(n_lanes, workers, [&](size_t lane, unsigned) {
#ifndef PPD_HOSTPROF
    CUDA_OK(cudaSetDevice(c->device));
#endif
    for (size_t i = lane; i < n; i += n_lanes) {
      decode_one(c, c->lanes[lane], flats[i], lens[i], &outs[i], &out_lens[i], &statuses[i], dump_workers);
      if (done) {  // streaming: the block's output goes to the caller now (and is the caller's to free)
        uint8_t* o = outs[i];
        outs[i] = nullptr;
        done(user, i, statuses[i], o, out_lens[i]);
      }
    }
  });
  c->last_lanes_used = n_lanes;
  for (size_t w = 0; w < n_lanes; w++) add_stats(c->stats, c->lanes[w]->stats);
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int ppd_ctx_create(int device, ppd_ctx** out) {
  if (!out) return PPD_ERR_BAD_ARGUMENT;
  *out = nullptr;
#ifdef PPD_HOSTPROF
  *out = new ppd_ctx();
  return PPD_OK;
#endif
  // every lane has its own stream; the device multiplexes streams onto CUDA_DEVICE_MAX_CONNECTIONS hardware queues
  // (8 unless set, 32 at most), and kernels of streams that share a queue wait for each other.  Only effective when
  // set before the process creates its CUDA context (lib.py and bench.py set it at import time for Python callers).
  setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return PPD_ERR_CUDA;
  ppd_ctx* c = new ppd_ctx();
  c->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) {
    delete c;
    return PPD_ERR_CUDA;
  }
  // the stream pool and the loop streams (host_pipeline.h: StreamPool): made first and together, so that they sit on
  // hardware queues of their own.  22 + 8 stay below the 32 queues.  In a sweep (profiles/r02b_knobs.txt: 512 config-2
  // blocks per stream call) 24 + 6 gave 619 blocks/s and 26 + 4 588, against two runs of 22 + 8 at 578 and 617.
  constexpr int MAIN_STREAMS = 22, LOOP_STREAMS = 8;
  c->pool = new StreamPool();
  for (int k = 0; k < MAIN_STREAMS; k++) {
    cudaStream_t s = nullptr;
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) {
      ppd_ctx_destroy(c);
      return PPD_ERR_CUDA;
    }
    c->pool->all.push_back(s), c->pool->free_.push_back(s);
  }
  c->batcher = loop_batcher_create(device, LOOP_STREAMS);
  if (!c->batcher) {
    ppd_ctx_destroy(c);
    return PPD_ERR_CUDA;
  }
  *out = c;
  return PPD_OK;
}

void ppd_ctx_destroy(ppd_ctx* c) {
  if (!c) return;
#ifdef PPD_HOSTPROF
  for (Lane* l : c->lanes) lane_delete(l);
  delete c;
  return;
#endif
  cudaSetDevice(c->device);
  if (c->batcher) loop_batcher_destroy(c->batcher);
  if (c->pool) {
    for (cudaStream_t s : c->pool->all) cudaStreamDestroy(s);
    delete c->pool;
  }
  for (Lane* l : c->lanes) lane_delete(l);
  DevBuf* bufs[] = {&c->d_keys, &c->d_vals, &c->d_ref, &c->d_ref_len, &c->d_counters, &c->d_msg, &c->d_msg_off, &c->d_digest};
  for (DevBuf* b : bufs) b->release();
  trie_release_all(c);
  c->build.release();
  for (DevBuf& b : c->d_leaves) b.release();
  for (DevBuf& b : c->d_subset) b.release();
  for (DevBuf& b : c->d_merge) b.release();
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->st) cudaStreamDestroy(c->st);
  delete c;
}

const char* ppd_last_error(const ppd_ctx* c) { return c ? c->err.c_str() : "null context"; }
void ppd_last_stats(const ppd_ctx* c, ppd_stats* out) {
  if (c && out) *out = c->stats;
}
void ppd_free(void* p) {
  if (p && !out_pool().give_back(p)) free(p);
}
void* ppd_alloc_pinned(size_t n) {
  void* p = out_pool().take(n ? n : 1);
  return p ? p : malloc(n ? n : 1);
}

int ppd_keccak256_batch(ppd_ctx* c, const uint8_t* data, const uint64_t* offsets, size_t n, uint8_t* out32n) {
  return guarded(c, [&] {
    stats_reset(c);
    if (!n) return;
    size_t bytes = offsets[n];
    c->d_msg.reserve(bytes + 16);
    c->d_msg_off.reserve((n + 1) * 8);
    c->d_digest.reserve(n * 32);
    CUDA_OK(cudaMemcpyAsync(c->d_msg.p, data, bytes, cudaMemcpyHostToDevice, c->st));
    CUDA_OK(cudaMemcpyAsync(c->d_msg_off.p, offsets, (n + 1) * 8, cudaMemcpyHostToDevice, c->st));
    CUDA_OK(cudaEventRecord(c->ev0, c->st));
    launch_keccak256_batch(c->d_msg.as<uint8_t>(), c->d_msg_off.as<uint64_t>(), (uint32_t)n, c->d_digest.as<uint8_t>(), c->st);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaEventRecord(c->ev1, c->st));
    CUDA_OK(cudaMemcpyAsync(out32n, c->d_digest.p, n * 32, cudaMemcpyDeviceToHost, c->st));
    CUDA_OK(cudaStreamSynchronize(c->st));
    float ms = 0;
    CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    c->stats.gpu_ms = ms;
    c->stats.key_hashes = n;
    for (size_t i = 0; i < n; i++) c->stats.key_permutations += (offsets[i + 1] - offsets[i]) / 136 + 1;
    c->stats.h2d_bytes = (double)(bytes + (n + 1) * 8);
    c->stats.d2h_bytes = (double)(n * 32);
    c->stats.kernel_launches = 1;
  });
}

// Measurement hooks: re-run kernels of the last ppd_block_decode / ppd_blocks_decode_batch call on what is still
// resident in HBM (no host work, no copies) and return the device time.  Every lane replays the selected stages in
// pipeline order on its own stream, lanes concurrently, as in the call itself:
//   PPD_REPLAY_PARSE  witness parse + pre-image arena (ppd_parse.cu)
//   PPD_REPLAY_HASH   key hashing and the level sweeps (ppd_kernels.cu); with TXN, the loop runs between the two sweeps
//   PPD_REPLAY_TXN    join (by root or by address), account table, op sort, the txn loop, the order of its nodes (ppd_txn.cu)
//   PPD_REPLAY_DUMP   IR sizing and emit (ppd_dump.cu)
// TXN and DUMP exist for lanes whose block took the device txn loop (gpu_txn.cu).
static void replay_lane(Lane* L, unsigned what) {
  cudaStream_t st = L->st;
  if ((what & PPD_REPLAY_PARSE) && L->has_last_parse) {
    ParseEmit E = L->last_emit;
    // the sweep may have moved the pools to larger buffers since
    E.nodes = L->d_nodes.as<NodeRec>(), E.key_pool = L->d_keys.as<uint8_t>(), E.val_pool = L->d_vals.as<uint8_t>();
    E.hash_pool = L->d_hashes.as<uint8_t>(), E.child_pool = L->d_children.as<uint32_t>(), E.accounts = L->d_accounts.as<AccountRec>();
    E.level = L->d_level.as<uint16_t>();
    CUDA_OK(cudaMemsetAsync(L->last_bounds.result, 0, 4 * PARSE_R_WORDS, st));
    launch_parse_bounds(L->last_bounds, st);
    launch_parse_scatter(L->last_bounds, L->last_ins_pos, st);
    launch_parse_tree(E.T, st);
    if (L->last_n_code) {
      launch_parse_code_list(E, st);
      launch_keccak256_ranges(E.T.wit, E.code_se, L->last_n_code, const_cast<uint8_t*>(E.code_digest), st);
    }
    if (L->last_val_bytes) CUDA_OK(cudaMemsetAsync(E.val_pool, 0, L->last_val_bytes, st));
    launch_parse_emit(E, st);
  }
  if ((what & PPD_REPLAY_HASH) && L->has_last) {
    CUDA_OK(cudaMemsetAsync(L->d_counters.p, 0, 32, st));
    if (L->last_msg_data)
      launch_keccak256_ranges(L->last_msg_data, L->last_msg_se, L->last_n_msgs, L->last_digest_out, st);
    else
      launch_keccak256_ranges(L->d_msg.as<uint8_t>(), L->d_msg_off.as<uint64_t>(), L->last_n_msgs, L->d_digest.as<uint8_t>(), st);
    for (size_t l = 0; l + 1 < L->last_level_start.size(); l++)
      launch_hash_level(L->last_view, L->d_order.as<uint32_t>(), L->last_level_start[l], L->last_level_start[l + 1], st);
  }
  if ((what & PPD_REPLAY_TXN) && L->has_last_txn) {
    const txn::View& v = L->last_txn;
    CUDA_OK(cudaMemsetAsync(v.touched, 0xff, 4ull * L->last_n_touched, st));
    CUDA_OK(cudaMemsetAsync(L->last_join.slot_owner, 0xff, 4ull * (L->last_join.table_mask + 1), st));
    CUDA_OK(cudaMemsetAsync(L->last_join.slot_best, 0, 4ull * (L->last_join.table_mask + 1), st));
    CUDA_OK(cudaMemsetAsync(v.pre_slot, 0xff, 4ull * (L->last_join.n_acct + 1), st));
    launch_txn_init(v, L->last_init, L->last_table_slots, st);
    if (L->last_join.keep)  // the lane's last block was a direct pre-image: its map's addresses are still resident
      launch_join_by_address(v, L->last_join, st);
    else
      launch_join(L->last_join, st);
    launch_txn_prep(v, L->last_ai, L->last_n_ops1, L->last_n_ops2, L->last_max_writes, st);
    launch_txn_loop(L->h_task, v, L->last_init.state_root, L->last_max_keys, st);
    CUDA_OK(cudaMemsetAsync(L->last_bins_tail, 0, 4ull * ORDER_MAX_BINS, st));
    launch_order_by_level_class(v.nodes, v.level, L->last_cap_tail, ORDER_MAX_BINS, L->last_okeys, L->last_bins_tail, L->d_order2.as<uint32_t>(), st,
                                L->last_init.n_nodes, &v.cur->n_nodes);
  }
  if ((what & PPD_REPLAY_HASH) && L->has_last) {
    // the nodes the device txn loop appended (gpu_txn.cu) are a second sweep over their own order
    for (size_t l = 0; l + 1 < L->last_level_start2.size(); l++)
      launch_hash_level(L->last_view, L->d_order2.as<uint32_t>(), L->last_level_start2[l], L->last_level_start2[l + 1], st);
  }
  if ((what & PPD_REPLAY_DUMP) && L->has_last_txn) {
    launch_ir_size(L->last_view, L->last_plan, L->last_n_ir, st);
    launch_ir_emit(L->last_view, L->last_plan, L->last_n_ir, L->d_out.as<uint8_t>(), st);
  }
  CUDA_OK(cudaGetLastError());
}

static const size_t REPLAY_LANES_MAX = 30;
size_t ppd_replay_lanes(const ppd_ctx* c) { return c ? std::min(std::min(c->last_lanes_used, c->lanes.size()), REPLAY_LANES_MAX) : 0; }
int ppd_replay_last(ppd_ctx* c, unsigned what, double* gpu_ms_out) {
  return guarded(c, [&] {
    size_t used = 0;
    const size_t n_lanes = ppd_replay_lanes(c);
    for (size_t w = 0; w < n_lanes; w++) {
      const Lane* L = c->lanes[w];
      used += ((what & PPD_REPLAY_PARSE) && L->has_last_parse) || ((what & PPD_REPLAY_HASH) && L->has_last) ||
              ((what & (PPD_REPLAY_TXN | PPD_REPLAY_DUMP)) && L->has_last_txn);
    }
    if (!used) fail(PPD_ERR_BAD_ARGUMENT, "nothing of the requested kind is resident");
    // all lanes start after ev0 on the main stream; the main stream then waits for every lane.  The calling thread
    // queues every lane: the replays are bound by the device, not by the queueing thread (profiles/r02b_replay_threads.txt:
    // 30 lanes' parse replay 13.4 ms queued by one thread, 13.7 ms by thirty; one thread launches 0.29 M kernels/s,
    // r02b_launch_rate.txt).
    CUDA_OK(cudaEventRecord(c->ev0, c->st));
    for (size_t w = 0; w < n_lanes; w++) {
      Lane* L = c->lanes[w];
      CUDA_OK(cudaStreamWaitEvent(L->st, c->ev0, 0));
      replay_lane(L, what);
      CUDA_OK(cudaEventRecord(L->ev1, L->st));
    }
    for (size_t w = 0; w < n_lanes; w++) CUDA_OK(cudaStreamWaitEvent(c->st, c->lanes[w]->ev1, 0));
    CUDA_OK(cudaEventRecord(c->ev1, c->st));
    CUDA_OK(cudaStreamSynchronize(c->st));
    float ms = 0;
    CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    if (gpu_ms_out) *gpu_ms_out = ms;
  });
}
int ppd_replay_last_hashing(ppd_ctx* c, double* gpu_ms_out) { return ppd_replay_last(c, PPD_REPLAY_HASH, gpu_ms_out); }
int ppd_replay_last_parse(ppd_ctx* c, double* gpu_ms_out) { return ppd_replay_last(c, PPD_REPLAY_PARSE, gpu_ms_out); }

// Measurement hook (ppd_microbench.cu): variant 0 = dependent-free LOP3/SHF issue rate, 1.. = register
// resident keccak-f variants.  units_out = ALU instructions (variant 0) or permutations executed.
int ppd_microbench(ppd_ctx* c, int variant, uint32_t blocks_per_sm, uint32_t iters, double* gpu_ms_out, double* units_out, uint32_t* digest_out) {
  return guarded(c, [&] {
    c->d_counters.reserve(64);
    CUDA_OK(cudaMemsetAsync(c->d_counters.p, 0, 64, c->st));
    uint32_t bt = 0;
    double per = 0;
    // warm-up launch, then the timed one
    if (!launch_microbench(variant, c->d_counters.as<uint32_t>(), blocks_per_sm, iters, &bt, &per, c->st)) fail(PPD_ERR_BAD_ARGUMENT, "unknown microbench variant");
    CUDA_OK(cudaEventRecord(c->ev0, c->st));
    launch_microbench(variant, c->d_counters.as<uint32_t>(), blocks_per_sm, iters, &bt, &per, c->st);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaEventRecord(c->ev1, c->st));
    uint32_t out[4];
    CUDA_OK(cudaMemcpyAsync(out, c->d_counters.p, 16, cudaMemcpyDeviceToHost, c->st));
    CUDA_OK(cudaStreamSynchronize(c->st));
    float ms = 0;
    CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    if (gpu_ms_out) *gpu_ms_out = ms;
    if (units_out) *units_out = per * (double)iters * (double)bt * 148.0 * (double)blocks_per_sm;
    if (digest_out) digest_out[0] = out[2], digest_out[1] = out[3];
  });
}

int ppd_compact_decode(ppd_ctx* c, const uint8_t* witness, size_t len, uint8_t** out, size_t* out_len) {
  return guarded(c, [&] {
    stats_reset(c);
    Lane* L = lane_of(c, 0);
    L->stats = ppd_stats{};
    Job& J = job_of(L, 1);
    BlockJob& b = J.blocks[0];
    if (len >= 0xffffffffull) fail(PPD_ERR_BAD_ARGUMENT, "witness larger than 4 GiB");
    b.compact = Span{witness, (uint32_t)len};
    if (!(gpu_parse_enabled() && gpu_pre_image(L, J, b, /*check_version=*/false))) {
      parse_witness(witness, len, b.wit);
      collect_witness_messages(J, b);
      J.kh.run(L);
      build_pre_image(J, b);
    }
    uint32_t sr = root_node_for(J, b, b.state_root);
    std::map<H256, uint32_t> storage_roots;
    b.storage.for_each([&](const H256Map::Entry& s) { storage_roots[s.first] = root_node_for(J, b, s.second); });
    sweep(L, J);
    c->stats = L->stats;
    Out o;
    o.u32(PPD_PRE_IMAGE_MAGIC);
    o.u8(b.wit.version);
    o.raw(J.ref.data() + 32ull * sr, 32);
    o.u32((uint32_t)storage_roots.size());
    for (auto& s : storage_roots) {
      o.raw(s.first.b, 32);
      o.raw(J.ref.data() + 32ull * s.second, 32);
    }
    o.u32((uint32_t)b.pre_code.size());
    for (auto& cd : b.pre_code) {
      o.raw(cd.first.b, 32);
      o.u32(cd.second.n);
    }
    o.u64(c->stats.nodes_hashed);
    o.u64(c->stats.node_permutations);
    *out = o.give(out_len);
  });
}

int ppd_blocks_decode_batch(ppd_ctx* c, const uint8_t* const* flats, const size_t* lens, size_t n, uint8_t** outs, size_t* out_lens,
                            int* statuses) {
  int rc = guarded(c, [&] { decode_blocks(c, flats, lens, n, outs, out_lens, statuses); });
  if (rc != PPD_OK && outs)  // a CUDA failure: no output is handed out (page-locked buffers go back to the pool)
    for (size_t i = 0; i < n; i++) {
      if (outs[i]) ppd_free(outs[i]);
      outs[i] = nullptr;
      if (out_lens) out_lens[i] = 0;
    }
  return rc;
}

int ppd_blocks_decode_stream(ppd_ctx* c, const uint8_t* const* flats, const size_t* lens, size_t n, ppd_block_done_fn done, void* user) {
  if (!done) return PPD_ERR_BAD_ARGUMENT;
  std::vector<uint8_t*> outs(n, nullptr);
  std::vector<size_t> out_lens(n, 0);
  std::vector<int> statuses(n, PPD_OK);
  int rc = guarded(c, [&] { decode_blocks(c, flats, lens, n, outs.data(), out_lens.data(), statuses.data(), done, user); });
  for (size_t i = 0; i < n; i++)  // (only after a failure: an output that was never handed over)
    if (outs[i]) ppd_free(outs[i]);
  return rc;
}

int ppd_block_decode(ppd_ctx* c, const uint8_t* flat, size_t len, uint8_t** out, size_t* out_len) {
  int status = PPD_OK;
  int rc = guarded(c, [&] { decode_blocks(c, &flat, &len, 1, out, out_len, &status); });
  if (rc != PPD_OK && out && *out) {
    ppd_free(*out);
    *out = nullptr;
  }
  return rc != PPD_OK ? rc : status;
}

}  // extern "C"
