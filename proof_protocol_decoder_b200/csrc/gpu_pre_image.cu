// gpu_pre_image.cu — host side of the witness parse + pre-image arena on the GPU (kernels: ppd_parse.cu).
#include "host_pipeline.h"

namespace ppd {

// ---- step 2 on the GPU (ppd_parse.cu): witness bytes -> instruction list -> tree links -> arena ------
// Three device phases with one small read-back each (instruction count; flags and pool sizes; the
// structural half of the arena).  The host keeps only what the txn loop walks (node records, keys,
// child lists, account records, levels); leaf values and the hashed-out subtrees stay in HBM.
// Returns false when the witness is not a well-formed canonical one: the host builder then takes it
// from the start and reports the reference's error, if any.
bool gpu_parse_enabled() {
#ifdef PPD_HOSTPROF
  return false;
#else
  return getenv("PPD_HOST_PARSE") == nullptr;  // read per call: the tests compare both builders in one process
#endif
}

struct Carve {
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

// Host bytes to the device on the lane's stream.  A page-locked caller buffer (ppd_alloc_pinned, cudaHostRegister) is
// read by the copy engine directly.  A pageable one is staged through the lane's page-locked buffer in chunks:
// concurrent pageable cudaMemcpyAsync calls serialise inside the driver, a plain memcpy per lane does not.
void upload_bytes(Lane* L, Job& J, uint8_t* dst, const uint8_t* src, size_t n) {
  cudaPointerAttributes at{};
  bool pinned = cudaPointerGetAttributes(&at, src) == cudaSuccess && at.type == cudaMemoryTypeHost;
  if (!pinned) cudaGetLastError();
  if (pinned) {
    CUDA_OK(cudaMemcpyAsync(dst, src, n, cudaMemcpyHostToDevice, L->st));
    return;
  }
  J.wit_stage.resize(n);
  const size_t CH = 4u << 20;
  for (size_t at0 = 0; at0 < n; at0 += CH) {
    size_t len = std::min(CH, n - at0);
    memcpy(J.wit_stage.data() + at0, src + at0, len);
    CUDA_OK(cudaMemcpyAsync(dst + at0, J.wit_stage.data() + at0, len, cudaMemcpyHostToDevice, L->st));
  }
}

bool gpu_pre_image(Lane* L, Job& J, BlockJob& b, bool check_version, Slots* slots, const PreImageDeviceOnly* dev_only) {
#ifdef PPD_HOSTPROF
  return false;
#else
  const uint8_t* w = b.compact.p;
  const size_t n = b.compact.n;
  if (n < 2 || n >= 0xfff00000ull) return false;
  // The three phases cost three read-backs and about 45 launches whatever the size: below a few hundred KiB
  // that latency exceeds what the host builder needs for the whole witness (config 4: 1024 blocks of 100 KB
  // each decode at 7.1 k blocks/s with the host builder, 3.3 k with this one), at config-2 size (36 MB) it
  // is 16x faster.  PPD_GPU_PARSE_MIN_BYTES moves the switch (the tests set it to 0).
  {
    const char* e = getenv("PPD_GPU_PARSE_MIN_BYTES");
    const size_t min_bytes = e ? (size_t)atoll(e) : (size_t)512 << 10;
    if (n < min_bytes) return false;
  }
  HostArena& A = J.A;
  cudaStream_t st = L->st;
  if (!L->h_parse) {
    L->h_parse = (uint32_t*)pinned_alloc(4 * PARSE_R_WORDS);
    if (!L->h_parse) fail(PPD_ERR_BAD_ARGUMENT, "out of page-locked memory");
  }
  uint32_t* hr = L->h_parse;
  static const bool timing = getenv("PPD_TIMING") != nullptr;
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!timing) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[ppd]   %-12s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_prev).count());
    t_prev = now;
  };
  // the waits while the slot is held sleep too: polling measured +3 % blocks/s for 3.5x the host CPU (DESIGN.md §3), and
  // polling threads of several GPUs' ranks would take cores from each other
  SlotGuard slot(slots, &L->stats.host_wait_ms);
  // the result words a host thread waits for: written into page-locked memory by a kernel when the whole block stays on
  // the device (a copy engine would serve them behind every bulk upload other lanes have queued)
  auto small_to_host = [&](void* dst, const void* src, size_t bytes) {
    if (!bytes) return;
    if (dev_only)
      lane_copy(L, dst, src, bytes);
    else
      CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
    L->stats.d2h_bytes += (double)bytes;
  };
  lap("p:slot-wait");
  trace_mark(L, "slot");
  // ---- phase A: instruction boundaries ----
  if (dev_only) {
    // the whole FlatBlock is resident (gpu_txn.cu uploaded it; the 64 bytes after it are zero)
  } else {
    L->d_wit.reserve(n + 64);
    upload_bytes(L, J, L->d_wit.as<uint8_t>(), w, n);
    CUDA_OK(cudaMemsetAsync(L->d_wit.as<uint8_t>() + n, 0, 64, st));
    L->stats.h2d_bytes += (double)n;
  }
  ParseBounds B{};
  auto result_to_host = [&] { small_to_host(hr, B.result, 4 * PARSE_R_WORDS); };
  B.wit = dev_only ? dev_only->d_witness : L->d_wit.as<uint8_t>();
  B.n = (uint32_t)n;
  B.n_tiles = (uint32_t)((n + PARSE_TILE - 1) / PARSE_TILE);
  B.group_tiles = 8;
  while (B.group_tiles < 1024 && (uint64_t)B.group_tiles * B.group_tiles < B.n_tiles) B.group_tiles *= 2;
  B.n_groups = (B.n_tiles + B.group_tiles - 1) / B.group_tiles;
  auto layout_a = [&](Carve& c) {
    B.result = c.take<uint32_t>(PARSE_R_WORDS);
    B.exit1 = c.take<uint32_t>((size_t)B.n_tiles * PARSE_TILE);  // whole tiles: tile_exit_kernel stores 128-bit rows
    B.step1 = c.take<uint16_t>((size_t)B.n_tiles * PARSE_TILE);
    B.exit2 = c.take<uint32_t>((size_t)B.n_groups * PARSE_TILE);
    B.group_entry = c.take<uint32_t>(B.n_groups);
    B.tile_entry = c.take<uint32_t>(B.n_tiles);
    B.bitmap = c.take<uint32_t>((size_t)B.n_tiles * (PARSE_TILE / 32));
    B.tile_count = c.take<uint32_t>(B.n_tiles + 1);
    B.tile_base = c.take<uint32_t>(B.n_tiles + 1);
    B.scan_tmp = c.take<uint32_t>(scan_tmp_words(B.n_tiles + 1));
  };
  {
    Carve sz{nullptr};
    layout_a(sz);
    L->d_pa.reserve(sz.off + 256);
    Carve c{L->d_pa.as<uint8_t>()};
    layout_a(c);
  }
  auto phase_ms = [&] {
    float ms = 0;
    CUDA_OK(cudaEventElapsedTime(&ms, L->ev0, L->ev1));
    L->stats.parse_gpu_ms += ms;
  };
  CUDA_OK(cudaMemsetAsync(B.result, 0, 4 * PARSE_R_WORDS, st));
  CUDA_OK(cudaEventRecord(L->ev0, st));
  L->stats.kernel_launches += launch_parse_bounds(B, st);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaEventRecord(L->ev1, st));
  result_to_host();
  lane_sync(L);
  phase_ms();
  lap("p:upload+A");
  trace_mark(L, "parse_a");
  if (hr[PARSE_R_END] != (uint32_t)n) return false;  // a parse error: the host parser reports it
  const uint32_t n_ins = hr[PARSE_R_NINS];
  if (n_ins == 0 || n_ins > n) return false;
  // phase B keeps about 100 bytes per instruction: a stream of one- and two-byte instructions (no real witness:
  // a node that can be a child is at least an opcode and a CBOR head) would ask for more memory than the witness
  // justifies; the host builder takes it
  if ((uint64_t)n_ins * 4 > (uint64_t)n + 256) return false;
  // ---- phase B: tree links, depths, sizes ----
  ParseTree T{};
  T.wit = B.wit, T.n = B.n, T.n_ins = n_ins, T.result = B.result;
  T.cnt_stride = ((size_t)n_ins + 1 + 3) & ~(size_t)3;
  uint32_t* ins_pos = nullptr;
  auto layout_b = [&](Carve& c) {
    const size_t n1 = (size_t)n_ins + 1;
    const size_t n_m1 = (n1 + 63) / 64, n_m2 = (n_m1 + 63) / 64, n_m3 = (n_m2 + 63) / 64;
    ins_pos = c.take<uint32_t>(n_ins);
    T.meta = c.take<uint32_t>(n_ins);
    T.knib = c.take<uint8_t>(n_ins);
    T.delta = c.take<uint32_t>(n1);
    T.hb = c.take<uint32_t>(n1);
    T.h16 = c.take<int16_t>(n1);
    T.m0 = c.take<int16_t>(8 * n_m1);
    T.m1 = c.take<int16_t>(n_m1);
    T.m2 = c.take<int16_t>(n_m2);
    T.m3 = c.take<int16_t>(n_m3);
    T.parent = c.take<uint32_t>(n_ins);
    T.info = c.take<uint32_t>(n_ins);
    T.aux0 = c.take<uint32_t>(n_ins);
    T.keyed = c.take<uint32_t>(n_ins);
    T.pending = c.take<uint32_t>(n_ins);
    T.lvlmax = c.take<uint32_t>(n_ins);
    T.cnt = c.take<uint32_t>(PARSE_N_CNT * T.cnt_stride);
    T.scn = c.take<uint32_t>(PARSE_N_CNT * T.cnt_stride);
    T.scan_tmp = c.take<uint32_t>(scan_tmp_words(n1, PARSE_N_CNT));
  };
  {
    Carve sz{nullptr};
    layout_b(sz);
    L->d_pb.reserve(sz.off + 256);
    Carve c{L->d_pb.as<uint8_t>()};
    layout_b(c);
  }
  T.ins_pos = ins_pos;
  CUDA_OK(cudaEventRecord(L->ev0, st));
  launch_parse_scatter(B, ins_pos, st);
  L->stats.kernel_launches += 1 + launch_parse_tree(T, st);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaEventRecord(L->ev1, st));
  result_to_host();
  lane_sync(L);
  phase_ms();
  lap("p:B");
  trace_mark(L, "parse_b");
  if (hr[PARSE_R_FLAG] != 0 || hr[PARSE_R_HEIGHT] != 1) return false;
  if (check_version && w[0] != 1) fail(PPD_PANIC_INCOMPATIBLE_HEADER_VERSION, "compact header version is not 1");
  const uint32_t* tot = hr + PARSE_R_TOTALS;
  const size_t n_nodes = tot[PARSE_C_NODE], n_hash = tot[PARSE_C_HASH], key_bytes = tot[PARSE_C_KEY], val_bytes = tot[PARSE_C_VAL],
               n_child = tot[PARSE_C_CHILD], n_acct = tot[PARSE_C_ACCT], n_code = tot[PARSE_C_CODE];
  const uint32_t root_ins = hr[PARSE_R_ROOT];
  if (root_ins >= n_ins || n_hash >= HASH_ID_END - HASH_ID_BASE) return false;
  // ---- phase C: emit the arena into the lane's buffers ----
  ParseEmit E{};
  E.T = T;
  E.n_keyed = hr[PARSE_R_NKEYED];
  if (E.n_keyed > n_ins) return false;
  uint16_t* d_level = nullptr;
  uint8_t* d_code_digest = nullptr;
  auto layout_c = [&](Carve& c) {
    E.acct_list = c.take<uint32_t>(5 * n_acct + 1);
    E.code_se = c.take<uint64_t>(2 * n_code + 1);
    E.code_list = c.take<uint32_t>(2 * n_code + 1);
    d_code_digest = c.take<uint8_t>(32 * n_code + 32);
  };
  {
    Carve sz{nullptr};
    layout_c(sz);
    L->d_pc.reserve(sz.off + 256);
    Carve c{L->d_pc.as<uint8_t>()};
    layout_c(c);
  }
  // room for what the txn loop appends, so that the sweep does not have to move the resident part
  if (dev_only) {
    const PreImageDeviceOnly& X = *dev_only;
    L->d_nodes.reserve(16 * (n_nodes + X.extra_nodes) + 4096);
    L->d_level.reserve(2 * (n_nodes + X.extra_nodes) + 4096);
    L->d_keys.reserve(key_bytes + X.extra_keys + 65536);
    L->d_vals.reserve(val_bytes + X.extra_vals + 65536);
    L->d_children.reserve(4 * (n_child + X.extra_children) + 4096);
    L->d_accounts.reserve(sizeof(AccountRec) * (n_acct + X.extra_accounts + 64));
  } else {
    L->d_nodes.reserve(16 * (n_nodes + n_nodes / 2) + 4096);
    L->d_level.reserve(2 * (n_nodes + n_nodes / 2) + 4096);
    L->d_keys.reserve(2 * key_bytes + 65536);
    L->d_vals.reserve(2 * val_bytes + 65536);
    L->d_children.reserve(4 * (n_child + n_child / 2) + 4096);
    L->d_accounts.reserve(sizeof(AccountRec) * (2 * n_acct + 64));
  }
  d_level = L->d_level.as<uint16_t>();
  L->d_hashes.reserve(32 * n_hash + 32);
  E.nodes = L->d_nodes.as<NodeRec>();
  E.level = d_level;
  E.key_pool = L->d_keys.as<uint8_t>();
  E.val_pool = L->d_vals.as<uint8_t>();
  E.hash_pool = L->d_hashes.as<uint8_t>();
  E.child_pool = L->d_children.as<uint32_t>();
  E.accounts = L->d_accounts.as<AccountRec>();
  E.code_digest = d_code_digest;
  CUDA_OK(cudaEventRecord(L->ev0, st));
  if (n_code) {
    launch_parse_code_list(E, st);
    launch_keccak256_ranges(B.wit, E.code_se, (uint32_t)n_code, d_code_digest, st);
    L->stats.kernel_launches += 2;
    L->stats.key_hashes += n_code;
  }
  if (val_bytes) CUDA_OK(cudaMemsetAsync(E.val_pool, 0, val_bytes, st));
  launch_parse_emit(E, st);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaEventRecord(L->ev1, st));
  L->stats.kernel_launches += 2;
  slot.done();  // the next lane may start its upload while this one's emit kernels and download run
  auto down = [&](void* dst, const void* src, size_t bytes) {
    if (!bytes) return;
    CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
    L->stats.d2h_bytes += (double)bytes;
  };
  J.code_list.resize(2 * n_code), J.code_digest.resize(n_code);
  if (!dev_only) {
    A.nodes.resize(n_nodes), A.level.resize(n_nodes), A.key_pool.resize(key_bytes), A.child_pool.resize(n_child), A.accounts.resize(n_acct);
    A.val_pool.resize(val_bytes), A.hash_pool.resize(32 * n_hash);  // contents stay on the device (fetch_pools)
    J.acct_list.resize(5 * n_acct);
    down(A.nodes.data(), E.nodes, 16 * n_nodes);
    down(A.level.data(), d_level, 2 * n_nodes);
    down(A.key_pool.data(), E.key_pool, key_bytes);
    down(A.child_pool.data(), E.child_pool, 4 * n_child);
    down(A.accounts.data(), E.accounts, sizeof(AccountRec) * n_acct);
    down(J.acct_list.data(), E.acct_list, 20 * n_acct);
  }
  small_to_host(J.code_list.data(), E.code_list, 8 * n_code);
  small_to_host(J.code_digest.data(), d_code_digest, 32 * n_code);
  result_to_host();
  lane_copy_flush(L);
  J.dev.nodes = n_nodes, J.dev.keys = key_bytes, J.dev.vals = val_bytes, J.dev.hashes = 32 * n_hash, J.dev.children = n_child, J.dev.accounts = n_acct;
  if (dev_only && dev_only->after_launch) dev_only->after_launch(dev_only->arg, E);  // queued behind the emit kernels, before the wait below
  lane_sync(L);
  phase_ms();
  lap("p:C+download");
  trace_mark(L, "parse_c");
  for (size_t k = 0; k < n_code; k++) {
    L->stats.key_permutations += J.code_list[2 * k + 1] / 136 + 1;
    b.pre_code[J.code_digest[k]] = Span{w + J.code_list[2 * k], J.code_list[2 * k + 1]};
  }
  J.pools_on_host = false;
  // ---- the block's per-account tables (compact_to_partial_trie.rs:167-190), as make_account_record builds them ----
  b.wit.version = w[0];
  b.state_root = hr[PARSE_R_ROOT_ID];
  if (dev_only) {  // the per-account tables are built on the device (ppd_txn.cu: join_*_kernel, acct_claim_kernel)
    b.pre_image_on_gpu = true;
    L->has_last_parse = true, L->last_bounds = B, L->last_emit = E, L->last_ins_pos = ins_pos, L->last_n_code = (uint32_t)n_code, L->last_val_bytes = val_bytes;
    L->stats.witnesses_on_gpu += 1, L->stats.witness_instructions += n_ins, L->stats.witness_bytes += n;
    return true;
  }
  b.storage.reserve(n_acct), b.pre_accounts.reserve(n_acct), b.root_of.reserve(2 * n_acct + 1024);
  b.have_empty_form = false, b.empty_form = NODE_EMPTY;
  const uint32_t* al = J.acct_list.data();
  for (size_t a = 0; a < n_acct; a++)
    if ((al[5 * a + 3] & 1u) && !(al[5 * a + 3] & 2u)) b.have_empty_form = true, b.empty_form = al[5 * a + 1];
  for (size_t a = 0; a < n_acct; a++) {
    const uint32_t leaf = al[5 * a], flags = al[5 * a + 3];
    const bool nonempty = flags & 2u;
    bool has_trie = flags & 1u;
    uint32_t sroot = al[5 * a + 1];
    if (!nonempty) has_trie = b.have_empty_form, sroot = b.empty_form;
    const NodeRec& nr = A.nodes[leaf];
    const uint32_t klen = ((nr.w0 >> 8) & 0xff) + ((nr.w0 >> 16) & 0xff);
    H256 haddr;
    if (klen == 64) {
      memcpy(haddr.b, A.key_pool.data() + nr.a0, 32);
    } else {  // utils.rs:49-59: the nibbles right-aligned in 32 bytes
      memset(haddr.b, 0, 32);
      for (uint32_t k = 0; k < klen; k++) {
        uint32_t posn = 64 - klen + k, nib = A.key_nib(nr.a0, k);
        haddr.b[posn >> 1] |= (uint8_t)((posn & 1) ? nib : (nib << 4));
      }
    }
    if (has_trie) b.storage[haddr] = sroot;
    b.pre_accounts.push_back({haddr, (uint32_t)a, nonempty, (flags & 1u) != 0, al[5 * a + 1]});
    if (nonempty) {
      b.pre_with_storage[haddr] = (uint32_t)a;
      b.root_of.put(al[5 * a + 1], al[5 * a + 2]);
    }
  }
  lap("p:tables");
  b.pre_image_on_gpu = true, b.pre_image_built = true;
  b.storage_partial = true;  // (not known without a pass over the arena: the join by root is always resolved)
  L->has_last_parse = true, L->last_bounds = B, L->last_emit = E, L->last_ins_pos = ins_pos, L->last_n_code = (uint32_t)n_code, L->last_val_bytes = val_bytes;
  L->stats.witnesses_on_gpu += 1, L->stats.witness_instructions += n_ins, L->stats.witness_bytes += n;
  if (getenv("PPD_VERIFY_GPU_PARSE")) verify_gpu_pre_image(L, J, b);
  return true;
#endif
}

// ---- PPD_VERIFY_GPU_PARSE: the GPU-built pre-image against the host builder's, node by node ----------
struct TrieCmp {
  const HostArena &X, &Y;
  std::string why;
  bool no(const char* what, uint32_t x, uint32_t y) {
    if (why.empty()) why = std::string(what) + " (gpu node " + std::to_string(x) + ", host node " + std::to_string(y) + ")";
    return false;
  }
  bool nibs_eq(uint32_t x, uint32_t y) {
    if (X.nstart(x) != Y.nstart(y) || X.nlen(x) != Y.nlen(y)) return false;
    for (uint32_t k = 0; k < X.nstart(x) + X.nlen(x); k++)  // the whole key up to the end of the node's range
      if (X.key_nib(X.nodes[x].a0, k) != Y.key_nib(Y.nodes[y].a0, k)) return false;
    return true;
  }
  bool eq(uint32_t x, uint32_t y) {
    if (x == NODE_EMPTY || y == NODE_EMPTY) return x == y ? true : no("empty vs non-empty", x, y);
    uint32_t kx = X.kind(x), ky = Y.kind(y);
    if (kx != ky) return no("node kinds differ", x, y);
    if (kx == NK_HASH) return memcmp(X.hash_of(x), Y.hash_of(y), 32) == 0 ? true : no("hashed-out nodes differ", x, y);
    if (X.lvl(x) != Y.lvl(y)) return no("levels differ", x, y);
    const NodeRec &a = X.nodes[x], &b = Y.nodes[y];
    switch (kx) {
      case NK_LEAF:
        if (!nibs_eq(x, y)) return no("leaf keys differ", x, y);
        if (a.a2 != b.a2 || memcmp(X.val_pool.data() + a.a1, Y.val_pool.data() + b.a1, a.a2) != 0) return no("leaf values differ", x, y);
        return true;
      case NK_LEAF_ACCOUNT: {
        if (!nibs_eq(x, y)) return no("account keys differ", x, y);
        const AccountRec &ra = X.accounts[a.a1], &rb = Y.accounts[b.a1];
        if (memcmp(&ra, &rb, 128) != 0) return no("account records differ", x, y);
        if ((ra.storage_src == NODE_EMPTY) != (rb.storage_src == NODE_EMPTY)) return no("account storage sources differ", x, y);
        return ra.storage_src == NODE_EMPTY ? true : eq(ra.storage_src, rb.storage_src);
      }
      case NK_EXT:
        if (!nibs_eq(x, y)) return no("extension keys differ", x, y);
        return eq(a.a1, b.a1);
      case NK_ROOT:
        return eq(a.a1, b.a1);
      case NK_BRANCH: {
        if ((a.a1 & 0xffff) != (b.a1 & 0xffff)) return no("branch masks differ", x, y);
        uint32_t k = (uint32_t)__builtin_popcount(a.a1 & 0xffff);
        for (uint32_t i = 0; i < k; i++)
          if (!eq(X.child_pool[a.a0 + i], Y.child_pool[b.a0 + i])) return false;
        return true;
      }
    }
    return no("unknown node kind", x, y);
  }
};

void verify_gpu_pre_image(Lane* L, Job& J, BlockJob& b) {
  fetch_pools(L, J);
  std::unique_ptr<Job> J2(new Job());
  J2->reset(1);
  BlockJob& b2 = J2->blocks[0];
  b2.compact = b.compact;
  parse_witness(b.compact.p, b.compact.n, b2.wit);
  collect_witness_messages(*J2, b2);
  J2->kh.run(L);
  build_pre_image(*J2, b2);
  auto bad = [&](const std::string& m) { throw Fail{PPD_ERR_CUDA, "GPU pre-image differs from the host builder's: " + m}; };
  TrieCmp cmp{J.A, J2->A};
  if (!cmp.eq(b.state_root, b2.state_root)) bad("state trie: " + cmp.why);
  if (b.storage.size() != b2.storage.size()) bad("storage map sizes " + std::to_string(b.storage.size()) + " / " + std::to_string(b2.storage.size()));
  b2.storage.for_each([&](const H256Map::Entry& s2) {
    auto f = b.storage.find(s2.first);
    if (f == b.storage.end()) bad("storage trie missing for an account");
    if (!cmp.eq(f->second, s2.second)) bad("storage trie: " + cmp.why);
  });
  if (b.pre_accounts.size() != b2.pre_accounts.size()) bad("pre-image account counts");
  for (size_t i = 0; i < b.pre_accounts.size(); i++) {
    const auto &p = b.pre_accounts[i], &q = b2.pre_accounts[i];
    if (!(p.haddr == q.haddr) || p.storage_nonempty != q.storage_nonempty || memcmp(&J.A.accounts[p.rec], &J2->A.accounts[q.rec], 128) != 0)
      bad("pre-image account " + std::to_string(i));
  }
  if (b.pre_with_storage.size() != b2.pre_with_storage.size()) bad("accounts with storage");
  b2.pre_with_storage.for_each([&](const H256Map::Entry& s2) {
    if (!b.pre_with_storage.count(s2.first)) bad("account with storage missing");
  });
  if (b.pre_code.size() != b2.pre_code.size()) bad("code map sizes");
  for (auto& c2 : b2.pre_code) {
    auto f = b.pre_code.find(c2.first);
    if (f == b.pre_code.end() || f->second.p != c2.second.p || f->second.n != c2.second.n) bad("code map entry");
  }
  b.root_of.for_each([&](uint32_t root, uint32_t root_node) {
    if (root_node >= J.A.nodes.size() || J.A.kind(root_node) != NK_ROOT || J.A.nodes[root_node].a1 != root) bad("root_of entry");
  });
}

}  // namespace ppd
