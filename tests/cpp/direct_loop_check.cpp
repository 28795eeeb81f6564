// tests/cpp/direct_loop_check.cpp — TEST INFRASTRUCTURE (CPU): the device txn loop on a direct pre-image (FlatBlock
// kind 2), with the device's by-address storage join (csrc/txn_core.h: join_addr_insert / join_addr_resolve), against
// the host path of the same block.  The companion of txn_core_check.cpp (kind 0, by-root join), whose node
// fingerprints (ArenaRO) and comparison this harness shares.
//
// Side 1 is the host path (ppd_host.cu: decode_one_inner): the pre-image re-spelled as a witness, the storage map cut to
// the addresses of the pre-image's map (direct_filter_storage), the host loop.  Side 2 runs the by-address join on the
// account list the GPU parser writes (built here from the host builder's tables), checks its arrays entry by entry
// against side 1's storage map, then runs the device loop with them and compares tries txn by txn.  Both sides build
// the pre-image with the same host builder, so their node ids agree.
//
// Built only by `make -C proof_protocol_decoder_b200/csrc directcheck` with -DPPD_HOSTPROF (no GPU, no node hashing).
//   build/directcheck <flat block file>...
#define main txn_core_check_main  // (the kind-0 harness's entry point; this file has its own)
#include "txn_core_check.cpp"
#undef main

namespace {

int check_direct_block(const std::vector<uint8_t>& flatv, const char* name) {
  const uint8_t* flat = flatv.data();
  // ---- side 1: the host txn loop ----
  Job J1;
  J1.reset(1);
  BlockJob& b1 = J1.blocks[0];
  read_flat_block(flat, flatv.size(), b1);
  if (b1.pre_image_kind != 2) {
    printf("%s: not a direct pre-image (kind %u)\n", name, b1.pre_image_kind);
    return 2;
  }
  PVec<uint8_t> wit1, wit2;
  direct_to_compact(b1, wit1);
  collect_messages(J1, b1);
  J1.kh.run(nullptr);
  // a block the host loop fails on (an error the reference reports) must never come out of the device path as a result:
  // the device side still runs, and has to decline the block or raise a flag (either hands the block to the host path)
  bool host_failed = false;
  Fail host_err{PPD_OK, ""};
  H256Map storage1;  // kind 2: the storage map the host path gives the loop (ppd_host.cu: decode_one_inner)
  try {
    build_pre_image(J1, b1);
    direct_filter_storage(b1);
    storage1 = b1.storage;
    shape_block(J1, b1);
  } catch (const Fail& e) {
    host_failed = true, host_err = e;
  }
  auto handed_over = [&](const char* how) {
    printf("%s: status %d (%s) from the host path; the device path %s\n", name, host_err.code, host_err.msg.c_str(), how);
    return 4;
  };
  // ---- side 2: the pre-image alone, then the device loop on host memory ----
  Job J2;
  J2.reset(1);
  BlockJob& b2 = J2.blocks[0];
  read_flat_block(flat, flatv.size(), b2);
  direct_to_compact(b2, wit2);
  collect_messages(J2, b2);
  J2.kh.run(nullptr);
  build_pre_image(J2, b2);
  HostArena& A = J2.A;
  TxnTables T;
  if (!txn_tables_phase1(b2, flat, flatv.size(), T)) {
    if (host_failed) return handed_over("declines the block in phase 1 of its tables");
    printf("%s: not a block the device loop takes: skipped\n", name);
    return 0;
  }
  const uint32_t n_traces = (uint32_t)T.traces.size();
  TxnBases B;
  B.dig_base = (uint32_t)((A.key_pool.size() + 31) & ~(size_t)31);
  B.txn_key_base = B.dig_base + 32 * T.n_msgs;
  B.key_cursor = B.txn_key_base + 12 * (uint32_t)b2.txns.size();
  B.val_base = (uint32_t)((A.val_pool.size() + 3) & ~(size_t)3);
  B.rec_base = (uint32_t)A.accounts.size();
  // memory of the "device"
  const uint32_t n_pre_nodes = (uint32_t)A.nodes.size();
  std::vector<NodeRec> nodes(n_pre_nodes + T.est_nodes);
  std::vector<uint16_t> level(nodes.size());
  memcpy(nodes.data(), A.nodes.data(), 16ull * n_pre_nodes);
  memcpy(level.data(), A.level.data(), 2ull * n_pre_nodes);
  std::vector<uint32_t> children(A.child_pool.size() + T.est_children);
  memcpy(children.data(), A.child_pool.data(), 4 * A.child_pool.size());
  std::vector<uint8_t> keys(B.key_cursor + 65536);
  memcpy(keys.data(), A.key_pool.data(), A.key_pool.size());
  std::vector<AccountRec> accounts(A.accounts.size() + T.n_recs + 1);
  memcpy(accounts.data(), A.accounts.data(), sizeof(AccountRec) * A.accounts.size());
  txn::View v;
  memset(&v, 0, sizeof v);
  v.nodes = nodes.data(), v.level = level.data(), v.key_pool = keys.data(), v.hash_pool = A.hash_pool.data();
  v.child_pool = children.data(), v.accounts = accounts.data();
  v.cap_nodes = (uint32_t)nodes.size(), v.cap_children = (uint32_t)children.size(), v.cap_keys = (uint32_t)keys.size();
  v.flat = flat, v.traces = T.traces.data(), v.n_txns = (uint32_t)b2.txns.size(), v.n_traces = n_traces, v.dig_base = B.dig_base;
  v.rec_base = B.rec_base, v.val_base = B.val_base;
  v.withdrawals = T.withdrawals.data(), v.n_withdrawals = (uint32_t)T.withdrawals.size();
  // digests (the device runs keccak256_batch_kernel over the same (begin, end) table)
  std::vector<uint64_t> se(2ull * T.n_msgs);
  for (uint32_t t = 0; t < n_traces; t++) txn::prep_msgs(v, t, se.data());
  for (uint32_t w = 0; w < v.n_withdrawals; w++) txn::prep_withdrawal_msg(v, w, se.data());
  for (uint32_t m = 0; m < T.n_msgs; m++) hostprof::keccak256(flat + se[2 * m], se[2 * m + 1] - se[2 * m], keys.data() + B.dig_base + 32ull * m);
  struct CD {
    txn::View* v;
    TxnTables* T;
  } cd{&v, &T};
  auto code_digest = [](void* arg, uint32_t t) -> const uint8_t* {
    CD* c = (CD*)arg;
    return c->v->key_pool + c->v->dig_base + 32ull * c->T->traces[t].m_code;
  };
  if (!txn_tables_phase2(b2, flat, B, code_digest, &cd, T)) {
    if (host_failed) return handed_over("declines the block in phase 2 of its tables");
    printf("%s: phase 2 declined the block (the host path reports its error): skipped\n", name);
    return 0;
  }
  memcpy(keys.data() + B.txn_key_base, T.txn_keys.data(), T.txn_keys.size());
  std::vector<uint8_t> vals(B.val_base + T.val_extra + 64);
  memcpy(vals.data(), A.val_pool.data(), A.val_pool.size());
  v.val_pool = vals.data();
  v.txns = T.txns.data();
  const uint32_t n_pre_acct = (uint32_t)A.accounts.size();
  std::vector<uint32_t> join_storage(n_pre_acct + 1, txn::ST_ABSENT), join_root(n_pre_acct + 1, txn::NONE);
  std::vector<uint8_t> pre_flags(n_pre_acct + 1, 0);
  int bad = 0;
  {
    // the by-address join of the device, on the account list the GPU parser writes (ppd_parse.cu: leaf node, storage
    // trie root, its NK_ROOT node, flags), here from the host builder's tables
    std::vector<uint32_t> acct_list(5ull * n_pre_acct + 5, 0);
    for (uint32_t n = 0; n < n_pre_nodes; n++)
      if ((A.nodes[n].w0 & 0xff) == NK_LEAF_ACCOUNT && A.nodes[n].a1 < n_pre_acct && !acct_list[5ull * A.nodes[n].a1 + 4])
        acct_list[5ull * A.nodes[n].a1] = n, acct_list[5ull * A.nodes[n].a1 + 4] = 1;
    for (const BlockJob::PreAccount& pa : b2.pre_accounts) {
      uint32_t* al = &acct_list[5ull * pa.rec];
      al[1] = pa.own_root;
      al[2] = pa.storage_nonempty ? A.accounts[pa.rec].storage_src : NODE_EMPTY;
      al[3] = (pa.witnesses_storage ? 1u : 0u) | (pa.storage_nonempty ? 2u : 0u);
    }
    uint32_t jtable = 64;
    while (jtable < 2 * std::max<size_t>(n_pre_acct, b2.direct_keep.size())) jtable <<= 1;
    std::vector<uint32_t> slot_owner(jtable, 0xffffffffu), slot_best(jtable, 0);
    txn::JoinView j;
    memset(&j, 0, sizeof j);
    j.acct_list = acct_list.data(), j.n_acct = n_pre_acct, j.slot_owner = slot_owner.data(), j.slot_best = slot_best.data();
    j.table_mask = jtable - 1, j.join_storage = join_storage.data(), j.join_root = join_root.data(), j.pre_flags = pre_flags.data();
    j.keep = reinterpret_cast<const uint8_t*>(b2.direct_keep.data());
    j.n_keep = (uint32_t)b2.direct_keep.size();
    for (uint32_t i = 0; i < std::max(j.n_keep, j.n_acct); i++) txn::join_addr_insert(j, i);
    for (uint32_t r = 0; r < n_pre_acct; r++) txn::join_addr_resolve(v, j, r);
    // entry by entry against the host path's storage map
    if (!host_failed) {
      for (size_t i = 0; i < b2.pre_accounts.size(); i++) {
        const BlockJob::PreAccount& pa = b2.pre_accounts[i];
        uint32_t want_s = txn::ST_ABSENT, want_r = txn::NONE;
        auto f = storage1.find(pa.haddr);
        if (f != storage1.end()) {
          want_s = f->second;
          if (const uint32_t* rn = b1.root_of.find(f->second)) want_r = *rn;
        }
        const bool same_acct = i < b1.pre_accounts.size() && b1.pre_accounts[i].haddr == pa.haddr && b1.pre_accounts[i].rec == pa.rec;
        if (!same_acct || join_storage[pa.rec] != want_s || join_root[pa.rec] != want_r || pre_flags[pa.rec] != (pa.storage_nonempty ? 1 : 0)) {
          if (bad++ < 10)
            printf("%s: by-address join of account %u: storage %x root %x flags %u, host path storage %x root %x flags %u\n", name, pa.rec, join_storage[pa.rec],
                   join_root[pa.rec], pre_flags[pa.rec], want_s, want_r, pa.storage_nonempty ? 1u : 0u);
        }
      }
    }
  }
  v.pre_flags = pre_flags.data();
  std::vector<uint32_t> pre_slot(n_pre_acct + 1, 0xffffffffu);
  v.pre_slot = pre_slot.data();
  uint32_t table = 64;
  while (table < 2 * n_traces) table <<= 1;
  std::vector<txn::AcctState> acct(table);
  memset(acct.data(), 0xff, sizeof(txn::AcctState) * table);
  v.acct = acct.data();
  std::vector<txn::SOp> ops1(T.n_ops1 + 1), ops2(T.n_ops2 + 1);
  v.ops1 = ops1.data(), v.ops2 = ops2.data();
  std::vector<uint32_t> touched(T.touched_begin.back() + 16, NODE_EMPTY);
  v.touched = touched.data(), v.seg_a = T.seg_a.data(), v.seg_b = T.seg_b.data();
  const size_t np = (size_t)T.max_ops * txn::PATH_CAP + 1;
  std::vector<uint32_t> path_node(np), path_pc(np), tnode(T.max_ops + 1), tpc(T.max_ops + 1), key_hi(T.max_ops + 1);
  std::vector<uint8_t> path_depth(np), plen(T.max_ops + 1), tdepth(T.max_ops + 1), tkind(T.max_ops + 1);
  std::vector<txn::SOp> sh_ops(T.max_ops + 1);
  v.s.path_node = path_node.data(), v.s.path_pc = path_pc.data(), v.s.path_depth = path_depth.data();
  v.s.plen = plen.data(), v.s.tnode = tnode.data(), v.s.tpc = tpc.data(), v.s.tdepth = tdepth.data(), v.s.tkind = tkind.data(), v.s.key_hi = key_hi.data();
  v.s.sh_ops = (n_traces & 1) ? sh_ops.data() : nullptr;  // both ways of reaching a txn's keys get exercised
  // the path-node table in two tiers, the first one tiny so that the spill tier is exercised
  std::vector<txn::PathNode> pc_fast(5), pc_slow(np);
  size_t map_n = 64;
  while (map_n < 2 * np) map_n <<= 1;
  std::vector<uint32_t> pc_map(map_n), pc_map_key(map_n);
  uint32_t pc_count = 0;
  v.s.pc_fast = pc_fast.data(), v.s.pc_n_fast = (uint32_t)pc_fast.size(), v.s.pc_slow = pc_slow.data(), v.s.pc_n_slow = (uint32_t)pc_slow.size();
  v.s.pc_map = pc_map.data(), v.s.pc_map_key = pc_map_key.data(), v.s.pc_map_mask = (uint32_t)map_n - 1, v.s.pc_count = &pc_count;
  txn::Cursors cur;
  memset(&cur, 0, sizeof cur);
  cur.n_nodes = n_pre_nodes, cur.n_children = (uint32_t)A.child_pool.size(), cur.key_bytes = B.key_cursor;
  cur.state_root = b2.state_root, cur.txn_root = NODE_EMPTY, cur.receipt_root = NODE_EMPTY;
  v.cur = &cur;
  v.s.a_nodes = &cur.n_nodes, v.s.a_children = &cur.n_children, v.s.a_keys = &cur.key_bytes, v.s.a_max_level = &cur.max_level;
  // ---- the kernels, in launch order ----
  txn::AcctInit ai{table - 1, b2.state_root, join_storage.data(), join_root.data()};
  for (uint32_t t = 0; t < n_traces; t++) txn::acct_claim(v, ai, t);
  for (uint32_t t = 0; t < n_traces; t++) txn::prep_trace(v, t);
  for (uint32_t t = 0; t < n_traces; t++)
    for (uint32_t k = 0; k < T.traces[t].n_keys; k++) txn::prep_storage_key(v, t, k);
  for (uint32_t ti = 0; ti < v.n_txns; ti++) txn::prep_txn(v, ti);
  for (uint32_t i = 0; i < T.n_ops1; i++) txn::prep_lcp(v, v.ops1, i);
  for (uint32_t i = 0; i < T.n_ops2; i++) txn::prep_lcp(v, v.ops2, i);
  long long sh_clock = 0;
  txn::Ctx c{v, 0, 1, &sh_clock};
  for (uint32_t ti = 0; ti < v.n_txns && !cur.flag; ti++) txn::run_txn(c, ti, EMPTY_TRIE_HASH, EMPTY_CODE_HASH);
  txn::run_finish(c, b2.state_root);
  if (host_failed) {
    if (cur.flag) {
      char how[96];
      snprintf(how, sizeof how, "raises flag %u at txn %u", cur.flag, cur.flag_txn);
      return handed_over(how);
    }
    printf("%s: MISMATCH: the device loop finished a block the host path fails with status %d (%s)\n", name, host_err.code, host_err.msg.c_str());
    return 1;
  }
  if (cur.flag) {
    printf("%s: the loop raised flag %u at txn %u (the host path would redo the block)\n", name, cur.flag, cur.flag_txn);
    return 2;
  }
  if (T.needs_dummies()) {
    // the storage map as the device exports it (ppd_txn.cu: acct_export_kernel)
    std::vector<txn::AcctExport> ex(n_pre_acct + 1);
    for (const BlockJob::PreAccount& pa : b2.pre_accounts) {
      txn::AcctExport e;
      memcpy(e.haddr, pa.haddr.b, 32);
      e.initial = join_storage[pa.rec];
      const uint32_t slot = pre_slot[pa.rec];
      e.final_ = slot < txn::NONE ? acct[slot].storage : e.initial;
      ex[pa.rec] = e;
    }
    txn_tables_dummies(b2, flat, cur, ex.data(), n_pre_acct, acct.data(), table, keys.data() + B.dig_base, T);
    v.seg_a = T.seg_a.data(), v.seg_b = T.seg_b.data();
  }
  // ---- the sweep's invariant: a node's level exceeds the level of everything it reads ----
  {
    auto lv = [&](uint32_t n) -> int { return (n == NODE_EMPTY || n >= 0x80000000u) ? -1 : (int)level[n]; };
    for (uint32_t n = n_pre_nodes; n < cur.n_nodes; n++) {
      const NodeRec r = nodes[n];
      const uint32_t kind = r.w0 & 0xff;
      int need = -1;
      if (kind == NK_EXT || kind == NK_ROOT) need = lv(r.a1);
      if (kind == NK_LEAF_ACCOUNT) need = lv(accounts[r.a1].storage_src);
      if (kind == NK_BRANCH)
        for (uint32_t j = 0; j < (uint32_t)__builtin_popcount(r.a1 & 0xffff); j++) need = std::max(need, lv(children[r.a0 + j]));
      if ((int)level[n] <= need) {
        printf("%s: node %u (kind %u) has level %u but reads a node of level %d\n", name, n, kind, level[n], need);
        return 1;
      }
    }
  }
  // ---- compare ----
  ArenaRO R1{J1.A.nodes.data(), J1.A.key_pool.data(), J1.A.val_pool.data(), J1.A.hash_pool.data(), J1.A.child_pool.data(), J1.A.accounts.data(), {}};
  ArenaRO R2{nodes.data(), keys.data(), vals.data(), A.hash_pool.data(), children.data(), accounts.data(), {}};
  auto expect = [&](bool ok, uint32_t ti, const char* what) {
    if (!ok && bad++ < 10) printf("%s: txn %u: %s differs\n", name, ti, what);
  };
  expect(b1.irs.size() == T.n_ir, 0, "number of IrDump entries");
  // dummy entries: the tries (roots only), every storage trie in hashed-address order, the roots after
  auto check_dummy = [&](int ir) {
    if (ir < 0 || (size_t)ir >= b1.irs.size()) return;
    IrPlan& p = b1.irs[ir];
    uint32_t q = T.seg_begin[ir];
    auto next_kind = [&](uint32_t kind) {
      while (q < T.seg_end[ir] && v.seg_b[q] != kind) q++;
      return q < T.seg_end[ir] ? q++ : 0xffffffffu;
    };
    uint32_t s0 = next_kind(IR_SEG_ROOT_ONLY), s1 = next_kind(IR_SEG_ROOT_ONLY), s2 = next_kind(IR_SEG_ROOT_ONLY);
    expect(s0 != 0xffffffffu && s2 != 0xffffffffu, ir, "dummy: trie segments");
    if (s2 == 0xffffffffu) return;
    expect(R1.fp(p.state_sub) == R2.fp(v.seg_a[s0]), ir, "dummy: state trie");
    expect(R1.fp(p.txn_sub) == R2.fp(v.seg_a[s1]), ir, "dummy: transactions trie");
    expect(R1.fp(p.receipt_sub) == R2.fp(v.seg_a[s2]), ir, "dummy: receipts trie");
    std::stable_sort(p.storage_subs.begin(), p.storage_subs.end(), [](const auto& x, const auto& y) { return x.first < y.first; });
    for (size_t k = 0; k < p.storage_subs.size(); k++) {
      uint32_t sq = next_kind(IR_SEG_ROOT_ONLY);
      expect(sq != 0xffffffffu, ir, "dummy: number of storage tries");
      if (sq == 0xffffffffu) return;
      // the hashed address is the tail of the literal segment before it
      const uint32_t lq = sq - 1;
      expect(v.seg_b[lq] == IR_SEG_LIT_DEV && memcmp(T.lit.data() + T.seg_c[lq] + v.seg_a[lq] - 32, p.storage_subs[k].first.b, 32) == 0, ir, "dummy: hashed address order");
      expect(R1.fp(p.storage_subs[k].second) == R2.fp(v.seg_a[sq]), ir, "dummy: a storage trie");
    }
    uint32_t r0 = next_kind(IR_SEG_REF), r1 = next_kind(IR_SEG_REF), r2 = next_kind(IR_SEG_REF);
    expect(r2 != 0xffffffffu, ir, "dummy: root segments");
    if (r2 == 0xffffffffu) return;
    expect(R1.fp(p.root_state) == R2.fp(v.seg_a[r0]), ir, "dummy: state root after");
    expect(R1.fp(p.root_txn) == R2.fp(v.seg_a[r1]), ir, "dummy: transactions root after");
    expect(R1.fp(p.root_receipt) == R2.fp(v.seg_a[r2]), ir, "dummy: receipts root after");
    bool has_wd_seg = false;
    for (uint32_t k = T.seg_begin[ir]; k < T.seg_end[ir]; k++)
      has_wd_seg |= v.seg_b[k] == IR_SEG_FLAT && !b2.withdrawals.empty() && T.seg_c[k] == (uint32_t)(b2.withdrawals[0].first - 4 - flat);
    expect(has_wd_seg == p.has_withdrawals, ir, "dummy: withdrawals");
  };
  check_dummy(T.dummy_initial[0]), check_dummy(T.dummy_initial[1]), check_dummy(T.dummy_final);
  for (uint32_t ti = 0; ti < v.n_txns; ti++) {
    IrPlan& p = b1.irs[T.first_txn_ir + ti];
    const txn::TxnDesc& tx = T.txns[ti];
    expect(R1.fp(p.state_sub) == R2.fp(v.seg_b[tx.seg_tries]), ti, "state trie before the txn");
    expect(R1.fp(p.txn_sub) == R2.fp(v.seg_b[tx.seg_tries + 1]), ti, "transactions trie before the txn");
    expect(R1.fp(p.receipt_sub) == R2.fp(v.seg_b[tx.seg_tries + 2]), ti, "receipts trie before the txn");
    std::stable_sort(p.storage_subs.begin(), p.storage_subs.end(), [](const auto& x, const auto& y) { return x.first < y.first; });
    const uint32_t ntr = tx.trace_end - tx.trace_begin;
    expect(p.storage_subs.size() == ntr, ti, "number of storage tries");
    for (uint32_t r = 0; r < ntr && r < p.storage_subs.size(); r++) {
      expect(v.seg_b[tx.seg_storage + 2 * r] == IR_SEG_KEY32, ti, "storage segment kind");
      expect(memcmp(keys.data() + v.seg_a[tx.seg_storage + 2 * r], p.storage_subs[r].first.b, 32) == 0, ti, "hashed address order");
      expect(R1.fp(p.storage_subs[r].second) == R2.fp(v.seg_b[tx.seg_storage + 2 * r + 1]), ti, "a storage trie before the txn");
    }
    expect(R1.fp(p.root_state) == R2.fp(v.seg_a[tx.seg_roots]), ti, "state trie after the txn");
    expect(R1.fp(p.root_txn) == R2.fp(v.seg_a[tx.seg_roots + 1]), ti, "transactions trie after the txn");
    expect(R1.fp(p.root_receipt) == R2.fp(v.seg_a[tx.seg_roots + 2]), ti, "receipts trie after the txn");
    std::set<uint64_t> t1, t2;
    for (uint32_t n : p.touched) t1.insert(R1.fp(n));
    for (uint32_t k = T.touched_begin[T.first_txn_ir + ti]; k < T.touched_begin[T.first_txn_ir + ti + 1]; k++)
      if (touched[k] != NODE_EMPTY) t2.insert(R2.fp(touched[k]));
    expect(t1 == t2, ti, "set of touched nodes");
  }
  printf("%s: %u txns, %u traces, %u + %u ops; host arena %zu nodes, device loop %u nodes (%u pre-image): %s\n", name, v.n_txns, n_traces, T.n_ops1,
         T.n_ops2, J1.A.nodes.size(), cur.n_nodes, n_pre_nodes, bad ? "MISMATCH" : "identical");
  return bad ? 1 : 0;
}

}  // namespace

int main(int argc, char** argv) {
  int rc = 0;
  for (int i = 1; i < argc; i++) {
    FILE* f = fopen(argv[i], "rb");
    if (!f) return 2;
    fseek(f, 0, SEEK_END);
    long n = ftell(f);
    fseek(f, 0, SEEK_SET);
    std::vector<uint8_t> flat(n);
    if (fread(flat.data(), 1, n, f) != (size_t)n) return 2;
    fclose(f);
    try {
      rc |= check_direct_block(flat, argv[i]);
    } catch (const Fail& e) {
      printf("%s: status %d (%s) from the host path\n", argv[i], e.code, e.msg.c_str());
      rc |= 4;
    }
  }
  return rc;
}
