// gpu_trie.cu — tries from leaves on the GPU (ppd_build.cu, ppd_leaves.cu, ppd_subset.cu, ppd_update.cu): the root and
// subset entries, which build a trie and drop it, and the trie handles, which keep one resident in HBM, cut subsets from
// it and update it in place (DESIGN.md §6).
#include "../../include/ppd_flat.h"
#include "host_pipeline.h"

using namespace ppd;

// ---- trie root over sorted leaves: structure built and hashed on the GPU (ppd_build.cu) ----------
namespace {

// The keys a trie subset is cut for (ppd_trie_subset_*): m device keys of key_len bytes, keccak256-hashed first when
// `hash`; the subset goes to *out / *out_len.
struct SubsetQuery {
  const uint8_t* d_keys;
  uint32_t key_len;
  bool hash;
  size_t m;
  uint8_t** out;
  size_t* out_len;
};
enum { SB_QKEYS, SB_BITS, SB_LIST, SB_SO, SB_SMALL, SB_OUT, SB_QRAW };

// create_trie_subset over the builder's arrays while they are resident (ppd_subset.cu).  end[]: the builder's branch bins
// (depth 63 - g owns bins 16 g .. 16 g + 15).  Leaves the subset in d_subset[SB_OUT] and returns its size.
size_t trie_subset_stage(ppd_ctx* c, const BuildView& V, uint32_t nb, const std::vector<uint32_t>& end, const SubsetQuery& q) {
  cudaStream_t st = c->st;
  const uint32_t n = V.n, m = (uint32_t)q.m;
  DevBuf* D = c->d_subset;
  SubsetView S;
  S.keys = V.keys, S.val_off = V.val_off, S.vals = V.vals, S.n = n, S.nb = nb;
  S.depth = V.depth, S.ext_start = V.ext_start, S.rep = V.rep, S.child = V.child, S.root_id = V.root_id;
  S.ref = V.ref, S.ref_len = V.ref_len, S.inner_ref = V.inner_ref, S.inner_ref_len = V.inner_ref_len;
  // a query touches at most one branch of each depth: depth d's bucket holds min(m, branches of depth d)
  uint32_t slots = 0;
  for (uint32_t d = 0; d < SUBSET_DEPTHS; d++) {
    const uint32_t g = 63 - d, bd = end[16 * g + 15] - (g ? end[16 * g - 1] : 0);
    S.base[d] = slots;
    slots += std::min(m, bd);
  }
  S.base[SUBSET_DEPTHS] = slots;
  const size_t bit_words = ((size_t)n + 2ull * nb + 31) / 32;
  D[SB_BITS].reserve(4 * bit_words);
  D[SB_LIST].reserve(4ull * slots + 64);
  D[SB_SO].reserve(8ull * nb + 64);
  D[SB_SMALL].reserve(512);  // [0, 64) counts, [64] flags, [66, 68) total
  S.bits = D[SB_BITS].as<uint32_t>(), S.list = D[SB_LIST].as<uint32_t>(), S.so = D[SB_SO].as<uint64_t>();
  uint32_t* small = D[SB_SMALL].as<uint32_t>();
  S.count = small, S.flags = small + 64, S.total = reinterpret_cast<unsigned long long*>(small + 66);
  CUDA_OK(cudaMemsetAsync(S.bits, 0, 4 * bit_words, st));
  CUDA_OK(cudaMemsetAsync(small, 0, 512, st));
  const uint8_t* q32 = q.d_keys;
  if (q.hash && m) {
    D[SB_QKEYS].reserve(32ull * m);
    launch_hash_fixed_keys(q.d_keys, q.key_len, m, D[SB_QKEYS].as<uint8_t>(), st);
    q32 = D[SB_QKEYS].as<uint8_t>();
    c->stats.key_hashes += m, c->stats.key_permutations += m, c->stats.kernel_launches += 1;
  } else if (m && (reinterpret_cast<uintptr_t>(q32) & 15)) {  // the walk loads each query as 16-byte words
    D[SB_QKEYS].reserve(32ull * m);
    CUDA_OK(cudaMemcpyAsync(D[SB_QKEYS].p, q32, 32ull * m, cudaMemcpyDeviceToDevice, st));
    q32 = D[SB_QKEYS].as<uint8_t>();
  }
  launch_subset_mark(S, q32, m, st);
  CUDA_OK(cudaGetLastError());
  uint32_t count[SUBSET_DEPTHS];
  CUDA_OK(cudaMemcpyAsync(count, small, sizeof count, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  uint32_t launches = m ? 3 : 2;
  for (uint32_t d = SUBSET_DEPTHS; d-- > 0;)
    if (count[d]) launch_subset_size(S, d, count[d], st), launches++;
  launch_subset_root(S, nullptr, false, st);
  CUDA_OK(cudaGetLastError());
  uint32_t tail[4];  // flags, (unused), total
  CUDA_OK(cudaMemcpyAsync(tail, small + 64, 16, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  if (tail[0] & SUBSET_F_DEEP) fail(PPD_ERR_CUDA, "internal error: an embedded subtree deeper than the subset's expansion stack");
  uint64_t total;
  memcpy(&total, tail + 2, 8);
  D[SB_OUT].reserve(total + 64);
  uint8_t* out = D[SB_OUT].as<uint8_t>();
  launch_subset_root(S, out, true, st);
  for (uint32_t d = 0; d < SUBSET_DEPTHS; d++)
    if (count[d]) launch_subset_emit(S, d, count[d], out, st), launches++;
  CUDA_OK(cudaGetLastError());
  c->stats.kernel_launches += launches;
  c->stats.d2h_bytes += sizeof count + 16;
  return total;
}

// the subset of trie_subset_stage, copied to a buffer the caller releases with ppd_free
void subset_to_host(ppd_ctx* c, size_t total, const SubsetQuery& q) {
  uint8_t* pinned = total >= ((size_t)1 << 20) ? out_pool().take(total) : nullptr;
  uint8_t* h = pinned ? pinned : (uint8_t*)malloc(total ? total : 1);
  if (!h) fail(PPD_ERR_BAD_ARGUMENT, "out of host memory for the subset");
  cudaError_t e = cudaMemcpyAsync(h, c->d_subset[SB_OUT].p, total, cudaMemcpyDeviceToHost, c->st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->st);
  if (e != cudaSuccess) {
    ppd_free(h);
    throw Fail{PPD_ERR_CUDA, std::string("subset copy: ") + cudaGetErrorString(e)};
  }
  c->stats.d2h_bytes += (double)total;
  *q.out = h, *q.out_len = total;
}

BuildView build_view(BuildState& S, const uint8_t* d_keys, const uint64_t* d_val_off, const uint8_t* d_vals, uint32_t n, uint32_t nb,
                     int base_depth, bool inner) {
  DevBuf* D = S.d;
  const uint32_t n1 = (n + 1 + 63) / 64, n2 = (n1 + 63) / 64;
  int8_t* m1 = D[BuildState::B_M].as<int8_t>();
  int8_t* m2 = m1 + ((n1 + 63) & ~63u);
  int8_t* m3 = m2 + ((n2 + 63) & ~63u);
  uint32_t* small = D[BuildState::B_SMALL].as<uint32_t>();
  BuildView V;
  V.keys = d_keys;
  V.val_off = d_val_off;
  V.vals = d_vals;
  V.n = n;
  V.base_depth = base_depth;
  V.P = Pyramid{D[BuildState::B_L].as<int8_t>(), m1, m2, m3};
  V.leader = D[BuildState::B_LINKA].as<uint32_t>();
  V.bidx = D[BuildState::B_BIDX].as<uint32_t>();
  V.depth = D[BuildState::B_DEPTH].as<uint8_t>();
  V.ext_start = V.depth + nb + 32;
  V.rep = D[BuildState::B_REP].as<uint32_t>();
  V.child = D[BuildState::B_CHILD].as<uint32_t>();
  V.root_id = small + 1;
  V.flags = small + 0;
  V.ref = D[BuildState::B_REF].as<uint8_t>();
  V.ref_len = D[BuildState::B_REF_LEN].as<uint8_t>();
  V.root_out = reinterpret_cast<uint8_t*>(small + 8);
  V.counters = reinterpret_cast<unsigned long long*>(small + 2);
  V.inner_ref = inner ? D[BuildState::B_IREF].as<uint8_t>() : nullptr;
  V.inner_ref_len = inner ? D[BuildState::B_IREF_LEN].as<uint8_t>() : nullptr;
  return V;
}

// The structure passes of the builder over n > 0 sorted leaves, into S: L, the pyramid, leaders, bidx, then every
// branch's depth, extension, rep and child table (leaves are placed by the leaf pass), and nchild.  `timed`: c->ev0 is
// recorded before the first pass.  inner: the view writes inner_ref (a subset is cut from the trie).
BuildView build_structure(ppd_ctx* c, BuildState& S, const uint8_t* d_keys, const uint64_t* d_val_off, const uint8_t* d_vals, uint32_t n,
                          int base_depth, bool inner, bool timed) {
  cudaStream_t st = c->st;
  const uint32_t n1 = (n + 1 + 63) / 64, n2 = (n1 + 63) / 64, n3 = (n2 + 63) / 64;
  DevBuf* D = S.d;
  D[BuildState::B_L].reserve((size_t)n + 1 + 64);
  D[BuildState::B_M].reserve((size_t)n1 + n2 + n3 + 192);
  D[BuildState::B_LINKA].reserve(4ull * (n + 1));
  D[BuildState::B_LINKB].reserve(4ull * (n + 1));
  D[BuildState::B_BIDX].reserve(4ull * (n + 1));
  D[BuildState::B_TMP].reserve(4ull * scan_tmp_words((size_t)n + 1));
  D[BuildState::B_SMALL].reserve(16384);
  BuildView V = build_view(S, d_keys, d_val_off, d_vals, n, 0, base_depth, false);
  const Pyramid P = V.P;
  // [0] error flags, [1] root id, [2..7] counters(u64 x 3), [8..15] root, [16] listed leaves, [32..95] marked
  // branches per depth (an update's), [1024..2111] branch bins
  uint32_t* small = D[BuildState::B_SMALL].as<uint32_t>();
  CUDA_OK(cudaMemsetAsync(small, 0, 16384, st));
  if (timed) CUDA_OK(cudaEventRecord(c->ev0, st));
  launch_lcp(d_keys, n, const_cast<int8_t*>(P.L), small + 0, st, base_depth);
  launch_min64(P.L, n + 1, const_cast<int8_t*>(P.m1), n1, st);
  launch_min64(P.m1, n1, const_cast<int8_t*>(P.m2), n2, st);
  launch_min64(P.m2, n2, const_cast<int8_t*>(P.m3), n3, st);
  uint32_t* leader = D[BuildState::B_LINKA].as<uint32_t>();
  uint32_t* flag = D[BuildState::B_LINKB].as<uint32_t>();
  launch_leaders(P.L, P.m1, P.m2, P.m3, n, leader, flag, flag, st);
  uint32_t* bidx = D[BuildState::B_BIDX].as<uint32_t>();
  exclusive_scan(flag, bidx, n + 1, D[BuildState::B_TMP].as<uint32_t>(), st);
  CUDA_OK(cudaGetLastError());
  uint32_t h_flags = 0, nb = 0;
  CUDA_OK(cudaMemcpyAsync(&h_flags, small, 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaMemcpyAsync(&nb, bidx + n, 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  if (h_flags & BUILD_F_UNSORTED) fail(PPD_ERR_UNSORTED_KEYS, "keys are not strictly ascending");
  if (h_flags & BUILD_F_PREFIX) fail(PPD_ERR_BAD_ARGUMENT, "the keys of a sub-trie do not share their first base_depth nibbles");
  c->stats.kernel_launches += 11 + 3;

  D[BuildState::B_DEPTH].reserve(2ull * nb + 64);
  D[BuildState::B_REP].reserve(4ull * nb + 64);
  D[BuildState::B_CHILD].reserve(64ull * nb + 64);
  D[BuildState::B_ORDER].reserve(4ull * nb + 64);
  D[BuildState::B_REF].reserve(32ull * ((size_t)n + nb));
  D[BuildState::B_REF_LEN].reserve((size_t)n + nb);
  if (inner) {
    D[BuildState::B_IREF].reserve(32ull * nb + 64);
    D[BuildState::B_IREF_LEN].reserve((size_t)nb + 64);
  }
  D[BuildState::B_NCHILD].reserve(4ull * nb + 64);
  D[BuildState::B_KEYS].reserve(2ull * nb + 64);
  V = build_view(S, d_keys, d_val_off, d_vals, n, nb, base_depth, inner);
  uint32_t* nchild = D[BuildState::B_NCHILD].as<uint32_t>();
  if (nb) CUDA_OK(cudaMemsetAsync(V.child, 0xff, 64ull * nb, st));
  if (nb) CUDA_OK(cudaMemsetAsync(nchild, 0, 4ull * nb, st));
  launch_branch_info(V, st);
  launch_child_count(leader, bidx, n, nchild, st);
  c->stats.kernel_launches += 2;
  S.n = n, S.nb = nb;
  return V;
}

// After the hashing: c->ev1, the root and the counters; the builder's flags checked.  levels: the launches of the
// branch levels, plus one.
void build_finish(ppd_ctx* c, const BuildState& S, uint32_t levels, uint8_t root_out[32]) {
  cudaStream_t st = c->st;
  const uint32_t* small = S.d[BuildState::B_SMALL].as<uint32_t>();
  CUDA_OK(cudaEventRecord(c->ev1, st));
  uint32_t out[16];
  CUDA_OK(cudaMemcpyAsync(out, small, 64, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  if (out[0] & BUILD_F_SHORT_TOP) fail(PPD_ERR_BAD_ARGUMENT, "the sub-trie's top node encodes to fewer than 32 bytes: its parent embeds it, not its hash");
  memcpy(root_out, out + 8, 32);
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  unsigned long long cnt[3];
  memcpy(cnt, out + 2, 24);
  c->stats.gpu_ms += ms;
  c->stats.nodes_hashed += cnt[0];
  c->stats.node_permutations += cnt[1];
  c->stats.node_bytes += cnt[2];
  c->stats.arena_nodes += (uint64_t)S.n + S.nb;
  c->stats.levels += levels;
  c->stats.d2h_bytes += 64 + 4096 + 8;
}

void empty_subset(const SubsetQuery& q) {
  uint8_t* h = (uint8_t*)malloc(1);
  if (!h) fail(PPD_ERR_BAD_ARGUMENT, "out of host memory for the subset");
  h[0] = PPD_NODE_EMPTY;
  *q.out = h, *q.out_len = 1;
}

// The whole build over n sorted leaves into S: structure, every leaf and branch hashed; then the subset stage when q is
// given.  inner: S keeps inner_ref (always with q).
void trie_root_sorted_dev(ppd_ctx* c, BuildState& S, const uint8_t* d_keys, const uint64_t* d_val_off, const uint8_t* d_vals, size_t n_,
                          uint8_t root_out[32], int base_depth = 0, const SubsetQuery* q = nullptr, bool inner = false) {
  if (n_ == 0) {
    memcpy(root_out, EMPTY_TRIE_HASH, 32);  // HashedPartialTrie::default().hash(): keccak(0x80), types.rs:30-34
    S.n = 0, S.nb = 0;
    if (q) empty_subset(*q);
    return;
  }
  if (n_ >= 0x7fffffffull) fail(PPD_ERR_BAD_ARGUMENT, "at most 2^31 - 2 leaves per call");
  const uint32_t n = (uint32_t)n_;
  cudaStream_t st = c->st;
  BuildView V = build_structure(c, S, d_keys, d_val_off, d_vals, n, base_depth, inner || q, true);
  const uint32_t nb = S.nb;
  uint32_t* small = S.d[BuildState::B_SMALL].as<uint32_t>();
  // counting sort by (depth, number of children), deepest depth first: the lanes of a warp walk the same number of
  // children and run the same number of permutations
  uint32_t* order = S.d[BuildState::B_ORDER].as<uint32_t>();
  launch_order_branches(V.depth, S.d[BuildState::B_NCHILD].as<uint32_t>(), nb, S.d[BuildState::B_KEYS].as<uint16_t>(), small + 1024, order, st);
  launch_hash_sorted_leaves(V, st);
  c->stats.kernel_launches += 4;
  std::vector<uint32_t>& end = S.end;  // end of every bucket: depth 63 - g owns buckets 16 g .. 16 g + 15
  end.resize(BRANCH_BINS);
  CUDA_OK(cudaMemcpyAsync(end.data(), small + 1024, 4 * BRANCH_BINS, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  if (end[BRANCH_BINS - 1] != nb) fail(PPD_ERR_CUDA, "branch histogram does not add up");
  uint32_t levels = 1;
  for (uint32_t g = 0, begin = 0; g < 64; g++) {
    const uint32_t e = end[16 * g + 15];
    if (e > begin) {
      launch_hash_branch_level(V, order, begin, e, st);
      c->stats.kernel_launches++;
      levels++;
    }
    begin = e;
  }
  CUDA_OK(cudaGetLastError());
  const size_t subset_bytes = q ? trie_subset_stage(c, V, nb, end, *q) : 0;
  build_finish(c, S, levels, root_out);
  if (q) subset_to_host(c, subset_bytes, *q);
}

// ---- trie root over leaves in any order (ppd_leaves.cu): sort, keep the last of each key, gather, then the builder ----

// byte digits of the n keys that take more than one value (bit p: digit p): the passes a sort cannot skip
uint32_t varying_digits(ppd_ctx* c, const uint64_t* keys, uint32_t n, uint32_t* counts) {
  CUDA_OK(cudaMemsetAsync(counts, 0, 8 * 256 * 4, c->st));
  launch_digit_counts(keys, n, counts, c->st);
  CUDA_OK(cudaGetLastError());
  std::vector<uint32_t> h(8 * 256);
  CUDA_OK(cudaMemcpyAsync(h.data(), counts, 8 * 256 * 4, cudaMemcpyDeviceToHost, c->st));
  CUDA_OK(cudaStreamSynchronize(c->st));
  c->stats.kernel_launches += 1;
  c->stats.d2h_bytes += 8 * 256 * 4;
  uint32_t mask = 0;
  for (int p = 0; p < 8; p++)
    if (std::find(h.begin() + 256 * p, h.begin() + 256 * (p + 1), n) == h.begin() + 256 * (p + 1)) mask |= 1u << p;
  return mask;
}

// stable LSD radix sort of the pairs (k[in][i], v[in][i]) by key over the digits of `digits`; k[1 - in] / v[1 - in] are the
// other halves of the ping-pong.  Returns which half holds the result.
int sort_pairs(ppd_ctx* c, uint64_t* const k[2], uint32_t* const v[2], int in, uint32_t n, uint32_t digits, uint32_t* hist, uint32_t* tmp) {
  for (int p = 0; p < 8; p++) {
    if (!(digits & (1u << p))) continue;
    c->stats.kernel_launches += launch_radix_pass(k[in], v[in], k[1 - in], v[1 - in], n, p, hist, hist + radix_hist_words(n), tmp, c->st);
    in = 1 - in;
  }
  CUDA_OK(cudaGetLastError());
  return in;
}

// the batch sorted, with the last occurrence of every key marked (sort_keep_last)
struct SortedLeaves {
  const uint8_t* keys32;  // the keys (hashed when the call hashes them), in input order
  uint32_t* idx;          // [n] input position of each sorted position
  uint32_t* keep;         // [n + 1] 1 at the last occurrence of a key; kpos: its exclusive scan
  uint32_t* kpos;
  uint64_t* koff;         // [n + 1] exclusive scan of the kept values' lengths
  uint32_t kept;
};
enum { B_HKEYS, B_K0, B_K1, B_V0, B_V1, B_V2, B_TIE, B_MEMBER, B_MPOS, B_START, B_SPOS, B_CPOS, B_CIDX, B_CRUN, B_CWORD,
       B_LEN, B_KOFF, B_HIST, B_TMP, B_TMP64, B_SMALL, B_OKEYS, B_OOFF, B_OVALS };

void check_key_form(uint32_t key_len, uint32_t flags) {
  if (flags & ~PPD_LEAVES_HASH_KEYS) fail(PPD_ERR_BAD_ARGUMENT, "unknown flag bits");
  const bool hash = flags & PPD_LEAVES_HASH_KEYS;
  if (hash ? (key_len < 1 || key_len > 135) : key_len != 32)
    fail(PPD_ERR_BAD_ARGUMENT, hash ? "hashed keys are 1 to 135 bytes long" : "keys are 32 bytes long unless PPD_LEAVES_HASH_KEYS is set");
}

// n > 0 leaves in any order (c->d_leaves): val_off checked, keys hashed under `hash`, sorted stably, the last of each
// key marked.  Records c->ev0 first; the caller records c->ev1 and adds the time.
SortedLeaves sort_keep_last(ppd_ctx* c, const uint8_t* d_keys, uint32_t key_len, bool hash, const uint64_t* d_val_off, uint32_t n,
                            size_t vals_bytes) {
  cudaStream_t st = c->st;
  DevBuf* D = c->d_leaves;
  const size_t hist_words = radix_hist_words(n);
  for (int b : {B_K0, B_K1, B_CWORD}) D[b].reserve(8ull * n);
  for (int b : {B_V0, B_V1, B_V2, B_CPOS, B_CIDX, B_CRUN}) D[b].reserve(4ull * n);
  for (int b : {B_TIE, B_MEMBER, B_MPOS, B_START, B_SPOS}) D[b].reserve(4ull * (n + 1));
  for (int b : {B_LEN, B_KOFF}) D[b].reserve(8ull * (n + 1));
  D[B_HIST].reserve(4 * 2 * hist_words);
  D[B_TMP].reserve(4 * scan_tmp_words(std::max<size_t>(hist_words, (size_t)n + 1)));
  D[B_TMP64].reserve(8 * scan_tmp_words((size_t)n + 1));
  D[B_SMALL].reserve(16384);
  uint32_t* small = D[B_SMALL].as<uint32_t>();  // [0] bad offsets, [1] ties, [2] members and [3] runs (read back), [1024..3071] digit counts
  uint32_t* hist = D[B_HIST].as<uint32_t>();
  uint32_t* tmp = D[B_TMP].as<uint32_t>();
  uint64_t* const K[2] = {D[B_K0].as<uint64_t>(), D[B_K1].as<uint64_t>()};
  uint32_t* tie = D[B_TIE].as<uint32_t>();
  CUDA_OK(cudaMemsetAsync(small, 0, 4096, st));
  CUDA_OK(cudaEventRecord(c->ev0, st));
  launch_check_offsets(d_val_off, n, vals_bytes, small + 0, st);
  const uint8_t* keys32 = d_keys;
  if (hash) {
    D[B_HKEYS].reserve(32ull * n);
    launch_hash_fixed_keys(d_keys, key_len, n, D[B_HKEYS].as<uint8_t>(), st);
    keys32 = D[B_HKEYS].as<uint8_t>();
    c->stats.key_hashes = n, c->stats.key_permutations = n, c->stats.kernel_launches += 1;
  }
  // the whole set on word 0: (word, input position) pairs
  launch_key_word(keys32, n, 0, K[0], D[B_V0].as<uint32_t>(), st);
  c->stats.kernel_launches += 2;
  uint32_t digits = varying_digits(c, K[0], n, small + 1024);
  uint32_t bad = 0;
  CUDA_OK(cudaMemcpyAsync(&bad, small + 0, 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  if (bad) fail(PPD_ERR_BAD_ARGUMENT, "val_off decreases somewhere or val_off[n] exceeds vals_bytes");
  uint32_t* const V01[2] = {D[B_V0].as<uint32_t>(), D[B_V1].as<uint32_t>()};
  const int r0 = sort_pairs(c, K, V01, 0, n, digits, hist, tmp);
  uint32_t* idx = V01[r0];  // input position of the element at each sorted position
  launch_tie_flags(K[r0], n, tie, small + 1, st);
  uint32_t ties = 0;
  CUDA_OK(cudaMemcpyAsync(&ties, small + 1, 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  c->stats.kernel_launches += 1;
  c->stats.d2h_bytes += 8;

  // refine the runs that tie on the words so far by the next word; runs keep their positions, so only their members move
  TieRuns R;
  R.member = D[B_MEMBER].as<uint32_t>(), R.mpos = D[B_MPOS].as<uint32_t>(), R.start = D[B_START].as<uint32_t>(), R.spos = D[B_SPOS].as<uint32_t>();
  R.cpos = D[B_CPOS].as<uint32_t>(), R.cidx = D[B_CIDX].as<uint32_t>(), R.crun = D[B_CRUN].as<uint32_t>(), R.cword = D[B_CWORD].as<uint64_t>();
  uint32_t* const VR[2] = {V01[1 - r0], D[B_V2].as<uint32_t>()};
  for (int w = 1; w < 4 && ties; w++) {
    launch_tie_members(tie, n, R.member, R.start, st);
    uint32_t scans = exclusive_scan(R.member, R.mpos, n + 1, tmp, st);
    scans += exclusive_scan(R.start, R.spos, n + 1, tmp, st);
    launch_tie_compact(R, keys32, idx, n, w, K[0], VR[0], st);
    CUDA_OK(cudaMemcpyAsync(small + 2, R.mpos + n, 4, cudaMemcpyDeviceToDevice, st));
    CUDA_OK(cudaMemcpyAsync(small + 3, R.spos + n, 4, cudaMemcpyDeviceToDevice, st));
    CUDA_OK(cudaMemsetAsync(small + 1, 0, 4, st));
    uint32_t mr[2];
    CUDA_OK(cudaMemcpyAsync(mr, small + 2, 8, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    const uint32_t m = mr[0], runs = mr[1];
    c->stats.kernel_launches += 2 + scans;
    c->stats.d2h_bytes += 8;
    // sort A: the members by the word; sort B: stably by run (the digits a run id below `runs` can have)
    const int ra = sort_pairs(c, K, VR, 0, m, varying_digits(c, K[0], m, small + 1024), hist, tmp);
    launch_tie_run_key(R, VR[ra], m, K[1 - ra], VR[1 - ra], st);
    uint32_t run_digits = 0;
    for (int p = 0; p < 4; p++)
      if ((uint64_t)(runs - 1) >> (8 * p)) run_digits |= 1u << p;
    const int rb = sort_pairs(c, K, VR, 1 - ra, m, run_digits, hist, tmp);
    launch_tie_writeback(R, VR[rb], m, idx, tie, small + 1, st);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(&ties, small + 1, 4, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    c->stats.kernel_launches += 2;
    c->stats.d2h_bytes += 4;
  }

  // the last occurrence of every key, packed: sorted keys32, offsets, values
  const uint32_t kept = n - ties;
  uint32_t* keep = R.member;
  uint32_t* kpos = R.mpos;
  uint64_t* len = D[B_LEN].as<uint64_t>();
  uint64_t* koff = D[B_KOFF].as<uint64_t>();
  launch_keep_last(tie, idx, d_val_off, n, keep, len, st);
  uint32_t scans = exclusive_scan(keep, kpos, n + 1, tmp, st);
  scans += exclusive_scan(len, koff, n + 1, D[B_TMP64].as<uint64_t>(), st);
  c->stats.kernel_launches += 2 + scans;
  return SortedLeaves{keys32, idx, keep, kpos, koff, kept};
}

// the kept leaves packed into d_leaves[B_OKEYS / B_OOFF / B_OVALS] (sorted keys32, offsets from 0, values)
void gather_leaves(ppd_ctx* c, const SortedLeaves& S, const uint64_t* d_val_off, const uint8_t* d_vals, uint32_t n, size_t vals_bytes) {
  DevBuf* D = c->d_leaves;
  D[B_OKEYS].reserve(32ull * S.kept);
  D[B_OOFF].reserve(8ull * (S.kept + 1));
  D[B_OVALS].reserve(vals_bytes + 64);  // the kept values add up to at most val_off[n] - val_off[0] <= vals_bytes
  launch_gather_leaves(S.keys32, S.idx, d_val_off, d_vals, n, S.keep, S.kpos, S.koff, D[B_OKEYS].as<uint8_t>(), D[B_OOFF].as<uint64_t>(),
                       D[B_OVALS].as<uint8_t>(), c->st);
  CUDA_OK(cudaGetLastError());
}

// c->ev0 .. c->ev1 into gpu_ms
void add_elapsed(ppd_ctx* c) {
  CUDA_OK(cudaEventRecord(c->ev1, c->st));
  CUDA_OK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  c->stats.gpu_ms += ms;
}

// sort, keep the last of each key, gather, then the whole build into S (the leaves stay in d_leaves[B_O*])
void trie_root_leaves_dev(ppd_ctx* c, BuildState& S, const uint8_t* d_keys, uint32_t key_len, uint32_t flags, const uint64_t* d_val_off,
                          const uint8_t* d_vals, size_t n_, size_t vals_bytes, uint8_t root_out[32], const SubsetQuery* q = nullptr,
                          bool inner = false) {
  check_key_form(key_len, flags);
  if (n_ == 0) {
    trie_root_sorted_dev(c, S, nullptr, nullptr, nullptr, 0, root_out, 0, q);
    return;
  }
  if (n_ >= 0x7fffffffull) fail(PPD_ERR_BAD_ARGUMENT, "at most 2^31 - 2 leaves per call");
  const uint32_t n = (uint32_t)n_;
  const SortedLeaves L = sort_keep_last(c, d_keys, key_len, (flags & PPD_LEAVES_HASH_KEYS) != 0, d_val_off, n, vals_bytes);
  gather_leaves(c, L, d_val_off, d_vals, n, vals_bytes);
  add_elapsed(c);  // the builder adds its own part
  DevBuf* D = c->d_leaves;
  try {
    trie_root_sorted_dev(c, S, D[B_OKEYS].as<uint8_t>(), D[B_OOFF].as<uint64_t>(), D[B_OVALS].as<uint8_t>(), L.kept, root_out, 0, q, inner);
  } catch (const Fail& f) {
    if (f.code != PPD_ERR_UNSORTED_KEYS) throw;
    fail(PPD_ERR_CUDA, "internal error: the sorted, de-duplicated leaves are not strictly ascending (a bug of the leaf sort, or device "
         "inputs that changed during the call)");
  }
}

}  // namespace

extern "C" {

int ppd_trie_root_sorted_leaves_dev(ppd_ctx* c, const uint8_t* d_keys32, const uint64_t* d_val_off, const uint8_t* d_vals, size_t n,
                                    size_t vals_bytes, uint8_t root_out[32]) {
  (void)vals_bytes;
  return guarded(c, [&] {
    stats_reset(c);
    trie_root_sorted_dev(c, c->build, d_keys32, d_val_off, d_vals, n, root_out);
  });
}

int ppd_trie_subroot_sorted_leaves_dev(ppd_ctx* c, const uint8_t* d_keys32, const uint64_t* d_val_off, const uint8_t* d_vals, size_t n,
                                       size_t vals_bytes, uint32_t base_depth, uint8_t ref_out[32]) {
  (void)vals_bytes;
  return guarded(c, [&] {
    stats_reset(c);
    if (base_depth >= 64 || n == 0) fail(PPD_ERR_BAD_ARGUMENT, "a sub-trie needs leaves and a base depth below 64");
    trie_root_sorted_dev(c, c->build, d_keys32, d_val_off, d_vals, n, ref_out, (int)base_depth);
  });
}

// The branch over up to 16 hashed children (the top of a trie whose sub-tries were hashed apart, on other streams or
// other GPUs): a three-node arena (16 hash-pool entries, the branch, its ROOT) through the ordinary level kernel.
int ppd_trie_root_from_children(ppd_ctx* c, const uint8_t* child_hashes16x32, uint32_t mask, uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    mask &= 0xffffu;
    if (__builtin_popcount(mask) < 2) fail(PPD_ERR_BAD_ARGUMENT, "a branch has at least two children");
    NodeRec nodes[2];
    uint32_t kids[16], k = 0;
    for (uint32_t i = 0; i < 16; i++)
      if (mask & (1u << i)) kids[k++] = HASH_ID_BASE + i;
    nodes[0] = NodeRec{node_w0(NK_BRANCH, 0, 0), 0, mask, 0};
    nodes[1] = NodeRec{node_w0(NK_ROOT, 0, 0), 0, 0, 0};
    c->d_keys.reserve(4096), c->d_vals.reserve(4096), c->d_ref.reserve(4096), c->d_ref_len.reserve(256), c->d_counters.reserve(32);
    c->d_msg.reserve(4096);  // hash pool, nodes, children
    uint8_t* base = c->d_msg.as<uint8_t>();
    CUDA_OK(cudaMemcpyAsync(base, child_hashes16x32, 512, cudaMemcpyHostToDevice, c->st));
    CUDA_OK(cudaMemcpyAsync(base + 512, nodes, sizeof nodes, cudaMemcpyHostToDevice, c->st));
    CUDA_OK(cudaMemcpyAsync(base + 1024, kids, 4 * k, cudaMemcpyHostToDevice, c->st));
    CUDA_OK(cudaMemsetAsync(c->d_counters.p, 0, 32, c->st));
    ArenaView V{};
    V.nodes = reinterpret_cast<const NodeRec*>(base + 512), V.hash_pool = base, V.child_pool = reinterpret_cast<const uint32_t*>(base + 1024);
    V.key_pool = c->d_keys.as<uint8_t>(), V.val_pool = c->d_vals.as<uint8_t>(), V.accounts = nullptr;
    V.ref = c->d_ref.as<uint8_t>(), V.ref_len = c->d_ref_len.as<uint8_t>(), V.counters = c->d_counters.as<unsigned long long>();
    launch_hash_level(V, nullptr, 0, 1, c->st);
    launch_hash_level(V, nullptr, 1, 2, c->st);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(root_out, V.ref + 32, 32, cudaMemcpyDeviceToHost, c->st));
    CUDA_OK(cudaStreamSynchronize(c->st));
    c->stats.nodes_hashed = 2, c->stats.kernel_launches = 2;
  });
}

int ppd_trie_root_sorted_leaves(ppd_ctx* c, const uint8_t* keys32, const uint64_t* val_off, const uint8_t* vals, size_t n,
                                uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    if (!n) {
      trie_root_sorted_dev(c, c->build, nullptr, nullptr, nullptr, 0, root_out);
      return;
    }
    size_t vb = val_off[n];
    c->d_keys.reserve(32 * n);
    c->d_msg_off.reserve(8 * (n + 1));
    c->d_vals.reserve(vb + 64);
    CUDA_OK(cudaMemcpyAsync(c->d_keys.p, keys32, 32 * n, cudaMemcpyHostToDevice, c->st));
    CUDA_OK(cudaMemcpyAsync(c->d_msg_off.p, val_off, 8 * (n + 1), cudaMemcpyHostToDevice, c->st));
    CUDA_OK(cudaMemcpyAsync(c->d_vals.p, vals, vb, cudaMemcpyHostToDevice, c->st));
    c->stats.h2d_bytes += (double)(32 * n + 8 * (n + 1) + vb);
    trie_root_sorted_dev(c, c->build, c->d_keys.as<uint8_t>(), c->d_msg_off.as<uint64_t>(), c->d_vals.as<uint8_t>(), n, root_out);
  });
}

int ppd_trie_root_leaves_dev(ppd_ctx* c, const uint8_t* d_keys, uint32_t key_len, uint32_t flags, const uint64_t* d_val_off, const uint8_t* d_vals,
                             size_t n, size_t vals_bytes, uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    trie_root_leaves_dev(c, c->build, d_keys, key_len, flags, d_val_off, d_vals, n, vals_bytes, root_out);
  });
}

int ppd_trie_root_leaves(ppd_ctx* c, const uint8_t* keys, uint32_t key_len, uint32_t flags, const uint64_t* val_off, const uint8_t* vals, size_t n,
                         uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    if (n && n < 0x7fffffffull && key_len >= 1 && key_len <= 135) {
      // upload, then the device path checks everything (the offsets included: vals_bytes is what the caller says val_off[n] is)
      const size_t vb = val_off[n];
      c->d_keys.reserve((size_t)key_len * n);
      c->d_msg_off.reserve(8 * (n + 1));
      c->d_vals.reserve(vb + 64);
      CUDA_OK(cudaMemcpyAsync(c->d_keys.p, keys, (size_t)key_len * n, cudaMemcpyHostToDevice, c->st));
      CUDA_OK(cudaMemcpyAsync(c->d_msg_off.p, val_off, 8 * (n + 1), cudaMemcpyHostToDevice, c->st));
      CUDA_OK(cudaMemcpyAsync(c->d_vals.p, vals, vb, cudaMemcpyHostToDevice, c->st));
      c->stats.h2d_bytes += (double)((size_t)key_len * n + 8 * (n + 1) + vb);
      trie_root_leaves_dev(c, c->build, c->d_keys.as<uint8_t>(), key_len, flags, c->d_msg_off.as<uint64_t>(), c->d_vals.as<uint8_t>(), n, vb, root_out);
    } else {
      trie_root_leaves_dev(c, c->build, nullptr, key_len, flags, nullptr, nullptr, n, 0, root_out);  // the empty trie, or the argument error
    }
  });
}

}  // extern "C"

// ---- create_trie_subset of the trie over leaves (ppd_subset.cu): the root entries above, then the subset stage ----
namespace {

SubsetQuery subset_query(const uint8_t* d_queries, uint32_t key_len, uint32_t flags, size_t m, uint8_t** out, size_t* out_len) {
  if (!out || !out_len) fail(PPD_ERR_BAD_ARGUMENT, "out and out_len are required");
  *out = nullptr, *out_len = 0;
  if (m >= 0x7ffffffeull) fail(PPD_ERR_BAD_ARGUMENT, "fewer than 2^31 - 2 query keys per call");
  if (m && !d_queries) fail(PPD_ERR_BAD_ARGUMENT, "no query keys");
  return SubsetQuery{d_queries, key_len, (flags & PPD_LEAVES_HASH_KEYS) != 0, m, out, out_len};
}

}  // namespace

extern "C" {

int ppd_trie_subset_leaves_dev(ppd_ctx* c, const uint8_t* d_keys, uint32_t key_len, uint32_t flags, const uint64_t* d_val_off, const uint8_t* d_vals,
                               size_t n, size_t vals_bytes, const uint8_t* d_queries, size_t m, uint8_t** out, size_t* out_len, uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    const SubsetQuery q = subset_query(d_queries, key_len, flags, m, out, out_len);
    trie_root_leaves_dev(c, c->build, d_keys, key_len, flags, d_val_off, d_vals, n, vals_bytes, root_out, &q);
  });
}

int ppd_trie_subset_leaves(ppd_ctx* c, const uint8_t* keys, uint32_t key_len, uint32_t flags, const uint64_t* val_off, const uint8_t* vals, size_t n,
                           const uint8_t* queries, size_t m, uint8_t** out, size_t* out_len, uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    SubsetQuery q = subset_query(queries, key_len, flags, m, out, out_len);
    if (key_len < 1 || key_len > 135) {  // the device path rejects it
      trie_root_leaves_dev(c, c->build, nullptr, key_len, flags, nullptr, nullptr, n, 0, root_out, &q);
      return;
    }
    if (m) {
      c->d_subset[SB_QRAW].reserve((size_t)key_len * m);
      CUDA_OK(cudaMemcpyAsync(c->d_subset[SB_QRAW].p, queries, (size_t)key_len * m, cudaMemcpyHostToDevice, c->st));
      c->stats.h2d_bytes += (double)((size_t)key_len * m);
      q.d_keys = c->d_subset[SB_QRAW].as<uint8_t>();
    }
    if (n && n < 0x7fffffffull) {
      const size_t vb = val_off[n];
      c->d_keys.reserve((size_t)key_len * n);
      c->d_msg_off.reserve(8 * (n + 1));
      c->d_vals.reserve(vb + 64);
      CUDA_OK(cudaMemcpyAsync(c->d_keys.p, keys, (size_t)key_len * n, cudaMemcpyHostToDevice, c->st));
      CUDA_OK(cudaMemcpyAsync(c->d_msg_off.p, val_off, 8 * (n + 1), cudaMemcpyHostToDevice, c->st));
      CUDA_OK(cudaMemcpyAsync(c->d_vals.p, vals, vb, cudaMemcpyHostToDevice, c->st));
      c->stats.h2d_bytes += (double)((size_t)key_len * n + 8 * (n + 1) + vb);
      trie_root_leaves_dev(c, c->build, c->d_keys.as<uint8_t>(), key_len, flags, c->d_msg_off.as<uint64_t>(), c->d_vals.as<uint8_t>(), n, vb, root_out, &q);
    } else {
      trie_root_leaves_dev(c, c->build, nullptr, key_len, flags, nullptr, nullptr, n, 0, root_out, &q);  // the empty trie, or the argument error
    }
  });
}

int ppd_trie_subset_sorted_leaves_dev(ppd_ctx* c, const uint8_t* d_keys32, const uint64_t* d_val_off, const uint8_t* d_vals, size_t n, size_t vals_bytes,
                                      const uint8_t* d_queries32, size_t m, uint8_t** out, size_t* out_len, uint8_t root_out[32]) {
  (void)vals_bytes;
  return guarded(c, [&] {
    stats_reset(c);
    const SubsetQuery q = subset_query(d_queries32, 32, 0, m, out, out_len);
    trie_root_sorted_dev(c, c->build, d_keys32, d_val_off, d_vals, n, root_out, 0, &q);
  });
}

}  // extern "C"

// ---- resident trie handles: create, subset, update (ppd_update.cu), destroy --------------------------------------------

// sorted, de-duplicated leaves: keys32, val_off (offsets into vals), vals
struct LeafSet {
  DevBuf keys, off, vals;
  void release() { keys.release(), off.release(), vals.release(); }
};

struct ppd_trie {
  ppd_ctx* ctx;
  uint32_t key_len, flags;
  BuildState st[2];  // st[cur]: the trie; the other: the spare an update builds into
  LeafSet leaves[2];
  int cur = 0;
  uint32_t n = 0;
  uint8_t root[32];
  void release() {
    for (BuildState& s : st) s.release();
    for (LeafSet& l : leaves) l.release();
  }
};

namespace {

enum { M_UPOS, M_WRITTEN, M_WPOS, M_DROP, M_DPOS, M_INS, M_IPOS, M_SRC, M_LEN, M_LIST, M_TMP, M_KEYS };

ppd_trie* checked(ppd_ctx* c, ppd_trie* t) {
  if (!t) fail(PPD_ERR_BAD_ARGUMENT, "no trie handle");
  if (t->ctx != c) fail(PPD_ERR_BAD_ARGUMENT, "the trie handle belongs to another context");
  return t;
}

// a new handle of c, built by `build` into its state 0 (leaves: its leaf set 0); registered with c once it succeeded
template <class F>
void trie_create(ppd_ctx* c, uint32_t key_len, uint32_t flags, ppd_trie** out, uint8_t root_out[32], F build) {
  if (!out) fail(PPD_ERR_BAD_ARGUMENT, "out is required");
  *out = nullptr;
  std::unique_ptr<ppd_trie> t(new ppd_trie{c, key_len, flags});
  try {
    build(*t);
  } catch (...) {
    t->release();
    throw;
  }
  c->tries.push_back(t.get());
  memcpy(root_out, t->root, 32);
  *out = t.release();
}

// The any-order creates: the one-shot path into the handle's state, which then takes over the gathered leaves.
void create_from_leaves(ppd_ctx* c, ppd_trie& t, const uint8_t* d_keys, uint32_t key_len, uint32_t flags, const uint64_t* d_val_off,
                        const uint8_t* d_vals, size_t n, size_t vals_bytes) {
  trie_root_leaves_dev(c, t.st[0], d_keys, key_len, flags, d_val_off, d_vals, n, vals_bytes, t.root, nullptr, true);
  t.n = t.st[0].n;
  if (t.n) {
    std::swap(t.leaves[0].keys, c->d_leaves[B_OKEYS]);
    std::swap(t.leaves[0].off, c->d_leaves[B_OOFF]);
    std::swap(t.leaves[0].vals, c->d_leaves[B_OVALS]);
  }
}

SubsetQuery handle_query(const ppd_trie& t, const uint8_t* queries, size_t m, uint8_t** out, size_t* out_len) {
  return subset_query(queries, t.key_len, t.flags, m, out, out_len);
}

void trie_subset(ppd_ctx* c, ppd_trie& t, const SubsetQuery& q) {
  if (!t.n) {
    empty_subset(q);
    return;
  }
  BuildState& S = t.st[t.cur];
  const LeafSet& L = t.leaves[t.cur];
  const BuildView V = build_view(S, L.keys.as<uint8_t>(), L.off.as<uint64_t>(), L.vals.as<uint8_t>(), S.n, S.nb, 0, true);
  CUDA_OK(cudaEventRecord(c->ev0, c->st));
  const size_t bytes = trie_subset_stage(c, V, S.nb, S.end, q);
  add_elapsed(c);
  subset_to_host(c, bytes, q);
}

// Applies the batch to t: sort and keep the last of each key, merge into the spare leaf set, build the structure into
// the spare state, copy the refs of the clean nodes and hash the rest; then swap.  Nothing of t changes before the swap.
void trie_update(ppd_ctx* c, ppd_trie& t, const uint8_t* d_keys, const uint8_t* d_del, const uint64_t* d_val_off, const uint8_t* d_vals,
                 size_t k_, size_t vals_bytes, uint8_t root_out[32]) {
  if (k_ >= 0x7ffffffeull) fail(PPD_ERR_BAD_ARGUMENT, "fewer than 2^31 - 2 updates per call");
  if (k_ == 0) {
    memcpy(root_out, t.root, 32);
    return;
  }
  if (!d_keys || !d_val_off) fail(PPD_ERR_BAD_ARGUMENT, "no keys or no value offsets");
  const uint32_t k = (uint32_t)k_, n_old = t.n;
  cudaStream_t st = c->st;
  DevBuf* D = c->d_merge;
  if (!(t.flags & PPD_LEAVES_HASH_KEYS) && (reinterpret_cast<uintptr_t>(d_keys) & 15)) {
    // the marking walk (subset_mark_kernel) loads 32-byte keys as 16-byte words: keys at any other alignment are staged
    D[M_KEYS].reserve(32ull * k);
    CUDA_OK(cudaMemcpyAsync(D[M_KEYS].p, d_keys, 32ull * k, cudaMemcpyDeviceToDevice, st));
    d_keys = D[M_KEYS].as<uint8_t>();
  }
  const SortedLeaves B = sort_keep_last(c, d_keys, t.key_len, (t.flags & PPD_LEAVES_HASH_KEYS) != 0, d_val_off, k, vals_bytes);
  add_elapsed(c);

  // merge
  CUDA_OK(cudaEventRecord(c->ev0, st));
  const LeafSet& O = t.leaves[t.cur];
  LeafSet& N = t.leaves[1 - t.cur];
  D[M_UPOS].reserve(4ull * k);
  D[M_WRITTEN].reserve(4ull * (k + 1));
  D[M_WPOS].reserve(4ull * (k + 1));
  for (int b : {M_DROP, M_DPOS, M_INS, M_IPOS}) D[b].reserve(4ull * (n_old + 2));
  D[M_TMP].reserve(8 * scan_tmp_words(std::max<size_t>((size_t)n_old + 2, (size_t)k + 1)));
  MergeView M{};
  M.ukeys32 = B.keys32, M.idx = B.idx, M.keep = B.keep, M.del = d_del, M.uoff = d_val_off, M.uvals = d_vals, M.k = k;
  M.okeys = O.keys.as<uint8_t>(), M.ooff = O.off.as<uint64_t>(), M.ovals = O.vals.as<uint8_t>(), M.n_old = n_old;
  M.upos = D[M_UPOS].as<uint32_t>(), M.written = D[M_WRITTEN].as<uint32_t>(), M.wpos = D[M_WPOS].as<uint32_t>();
  M.drop = D[M_DROP].as<uint32_t>(), M.dpos = D[M_DPOS].as<uint32_t>(), M.ins = D[M_INS].as<uint32_t>(), M.ipos = D[M_IPOS].as<uint32_t>();
  CUDA_OK(cudaMemsetAsync(M.drop, 0, 4ull * (n_old + 2), st));
  CUDA_OK(cudaMemsetAsync(M.ins, 0, 4ull * (n_old + 2), st));
  launch_merge_locate(M, st);
  uint32_t* tmp = D[M_TMP].as<uint32_t>();
  uint32_t scans = exclusive_scan(M.written, M.wpos, k + 1, tmp, st);
  scans += exclusive_scan(M.drop, M.dpos, n_old + 1, tmp, st);
  scans += exclusive_scan(M.ins, M.ipos, n_old + 2, tmp, st);
  CUDA_OK(cudaGetLastError());
  uint32_t counts[2];
  CUDA_OK(cudaMemcpyAsync(counts, M.wpos + k, 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaMemcpyAsync(counts + 1, M.dpos + n_old, 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  const uint64_t n_new64 = (uint64_t)n_old - counts[1] + counts[0];
  if (n_new64 >= 0x7ffffffeull) fail(PPD_ERR_BAD_ARGUMENT, "the update would leave 2^31 - 2 or more leaves");
  const uint32_t n_new = (uint32_t)n_new64;
  M.n_new = n_new;
  D[M_SRC].reserve(4ull * n_new + 64);
  D[M_LEN].reserve(8ull * (n_new + 1));
  D[M_TMP].reserve(8 * scan_tmp_words((size_t)n_new + 1));  // the scan of len: a batch may grow the trie past n_old + 2 and k + 1
  N.off.reserve(8ull * (n_new + 1));
  N.keys.reserve(32ull * n_new + 64);
  M.src = D[M_SRC].as<uint32_t>(), M.len = D[M_LEN].as<uint64_t>(), M.noff = N.off.as<uint64_t>(), M.nkeys = N.keys.as<uint8_t>();
  launch_merge_place(M, st);
  scans += exclusive_scan(M.len, M.noff, n_new + 1, D[M_TMP].as<uint64_t>(), st);
  uint64_t vbytes = 0;
  CUDA_OK(cudaMemcpyAsync(&vbytes, M.noff + n_new, 8, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  N.vals.reserve(vbytes + 64);
  M.nvals = N.vals.as<uint8_t>();
  launch_merge_copy(M, st);
  CUDA_OK(cudaGetLastError());
  c->stats.kernel_launches += 3 + scans;
  c->stats.d2h_bytes += 16;

  uint8_t root[32];
  BuildState& S = t.st[1 - t.cur];
  if (n_new == 0) {
    add_elapsed(c);
    memcpy(root, EMPTY_TRIE_HASH, 32);
    S.n = 0, S.nb = 0;
  } else {
    const BuildState& P = t.st[t.cur];
    OldTrie OT{};
    OT.n = n_old;
    if (n_old) {
      const BuildView PV = build_view(const_cast<BuildState&>(P), nullptr, nullptr, nullptr, n_old, P.nb, 0, true);
      OT.L = PV.P.L, OT.leader = PV.leader, OT.bidx = PV.bidx, OT.depth = PV.depth, OT.ext_start = PV.ext_start;
      OT.ref = PV.ref, OT.ref_len = PV.ref_len, OT.inner_ref = PV.inner_ref, OT.inner_ref_len = PV.inner_ref_len;
    }
    const BuildView V = build_structure(c, S, N.keys.as<uint8_t>(), N.off.as<uint64_t>(), N.vals.as<uint8_t>(), n_new, 0, true, false);
    const uint32_t nb = S.nb;
    uint32_t* small = S.d[BuildState::B_SMALL].as<uint32_t>();
    // leaves: clean ones copy their refs, the rest are listed and hashed
    D[M_LIST].reserve(4ull * n_new + 64);
    launch_update_leaves(V, OT, M.src, D[M_LIST].as<uint32_t>(), small + 16, st);
    // branches: the batch's keys mark the branches whose prefix they share (the subset's marking walk)
    DevBuf* Q = c->d_subset;
    const size_t bit_words = ((size_t)n_new + 2ull * nb + 31) / 32;
    Q[SB_BITS].reserve(4 * bit_words);
    CUDA_OK(cudaMemsetAsync(Q[SB_BITS].p, 0, 4 * bit_words, st));
    SubsetView SV{};
    SV.keys = V.keys, SV.val_off = V.val_off, SV.vals = V.vals, SV.n = n_new, SV.nb = nb;
    SV.depth = V.depth, SV.ext_start = V.ext_start, SV.rep = V.rep, SV.child = V.child, SV.root_id = V.root_id;
    SV.bits = Q[SB_BITS].as<uint32_t>(), SV.count = small + 32;  // every depth's bucket is empty: nothing is listed
    launch_subset_mark(SV, B.keys32, k, st);
    uint32_t* nchild = S.d[BuildState::B_NCHILD].as<uint32_t>();
    launch_update_branches(V, OT, M.src, SV.bits, nchild, st);
    uint32_t* order = S.d[BuildState::B_ORDER].as<uint32_t>();
    launch_order_update_branches(V.depth, nchild, nb, S.d[BuildState::B_KEYS].as<uint16_t>(), small + 1024, order, st);
    CUDA_OK(cudaGetLastError());
    std::vector<uint32_t> bins(UPDATE_BRANCH_BINS);
    uint32_t listed = 0;
    CUDA_OK(cudaMemcpyAsync(&listed, small + 16, 4, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaMemcpyAsync(bins.data(), small + 1024, 4 * UPDATE_BRANCH_BINS, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    if (bins[UPDATE_BRANCH_BINS - 1] != nb) fail(PPD_ERR_CUDA, "branch histogram does not add up");
    launch_hash_listed_leaves(V, D[M_LIST].as<uint32_t>(), listed, st);
    c->stats.kernel_launches += 1 + 1 + 1 + 3 + (listed ? 1 : 0);
    // the branches to hash, deepest depth first; S.end: every depth's total, hashed and copied (the subset's bins)
    uint32_t levels = 1;
    S.end.assign(BRANCH_BINS, 0);
    for (uint32_t g = 0, begin = 0, all = 0; g < 64; g++) {
      const uint32_t e = bins[16 * g + 15];
      if (e > begin) {
        launch_hash_branch_level(V, order, begin, e, st);
        c->stats.kernel_launches++;
        levels++;
      }
      all += (e - begin) + bins[BRANCH_BINS + g] - (bins[BRANCH_BINS + g - 1]);
      for (uint32_t j = 0; j < 16; j++) S.end[16 * g + j] = all;
      begin = e;
    }
    CUDA_OK(cudaGetLastError());
    c->stats.d2h_bytes += 4 + 4 * UPDATE_BRANCH_BINS;
    build_finish(c, S, levels, root);
  }
  // everything succeeded: the spare becomes the trie
  t.cur = 1 - t.cur;
  t.n = n_new;
  memcpy(t.root, root, 32);
  memcpy(root_out, root, 32);
}

}  // namespace

namespace ppd {
void trie_release_all(ppd_ctx* c) {
  for (ppd_trie* t : c->tries) {
    t->release();
    delete t;
  }
  c->tries.clear();
}
}  // namespace ppd

extern "C" {

int ppd_trie_create_leaves_dev(ppd_ctx* c, const uint8_t* d_keys, uint32_t key_len, uint32_t flags, const uint64_t* d_val_off, const uint8_t* d_vals,
                               size_t n, size_t vals_bytes, ppd_trie** out, uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    trie_create(c, key_len, flags, out, root_out,
                [&](ppd_trie& t) { create_from_leaves(c, t, d_keys, key_len, flags, d_val_off, d_vals, n, vals_bytes); });
  });
}

int ppd_trie_create_leaves(ppd_ctx* c, const uint8_t* keys, uint32_t key_len, uint32_t flags, const uint64_t* val_off, const uint8_t* vals, size_t n,
                           ppd_trie** out, uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    trie_create(c, key_len, flags, out, root_out, [&](ppd_trie& t) {
      if (n && n < 0x7fffffffull && key_len >= 1 && key_len <= 135) {
        const size_t vb = val_off[n];
        c->d_keys.reserve((size_t)key_len * n);
        c->d_msg_off.reserve(8 * (n + 1));
        c->d_vals.reserve(vb + 64);
        CUDA_OK(cudaMemcpyAsync(c->d_keys.p, keys, (size_t)key_len * n, cudaMemcpyHostToDevice, c->st));
        CUDA_OK(cudaMemcpyAsync(c->d_msg_off.p, val_off, 8 * (n + 1), cudaMemcpyHostToDevice, c->st));
        CUDA_OK(cudaMemcpyAsync(c->d_vals.p, vals, vb, cudaMemcpyHostToDevice, c->st));
        c->stats.h2d_bytes += (double)((size_t)key_len * n + 8 * (n + 1) + vb);
        create_from_leaves(c, t, c->d_keys.as<uint8_t>(), key_len, flags, c->d_msg_off.as<uint64_t>(), c->d_vals.as<uint8_t>(), n, vb);
      } else {
        create_from_leaves(c, t, nullptr, key_len, flags, nullptr, nullptr, n, 0);  // the empty trie, or the argument error
      }
    });
  });
}

int ppd_trie_create_sorted_leaves_dev(ppd_ctx* c, const uint8_t* d_keys32, const uint64_t* d_val_off, const uint8_t* d_vals, size_t n,
                                      size_t vals_bytes, ppd_trie** out, uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    trie_create(c, 32, 0, out, root_out, [&](ppd_trie& t) {
      if (n >= 0x7fffffffull) fail(PPD_ERR_BAD_ARGUMENT, "at most 2^31 - 2 leaves per call");
      LeafSet& L = t.leaves[0];
      if (n) {
        // the handle builds and later merges from its own copy of vals_bytes bytes: val_off must stay inside them
        DevBuf& flag = c->d_leaves[B_SMALL];
        flag.reserve(16384);
        uint32_t bad = 0;
        CUDA_OK(cudaMemsetAsync(flag.p, 0, 4, c->st));
        launch_check_offsets(d_val_off, (uint32_t)n, vals_bytes, flag.as<uint32_t>(), c->st);
        CUDA_OK(cudaGetLastError());
        CUDA_OK(cudaMemcpyAsync(&bad, flag.p, 4, cudaMemcpyDeviceToHost, c->st));
        CUDA_OK(cudaStreamSynchronize(c->st));
        c->stats.kernel_launches += 1;
        if (bad) fail(PPD_ERR_BAD_ARGUMENT, "val_off decreases somewhere or val_off[n] exceeds vals_bytes");
      }
      if (n) {  // the caller's buffers are only borrowed for the call: the handle keeps a copy
        L.keys.reserve(32ull * n + 64);
        L.off.reserve(8ull * (n + 1));
        L.vals.reserve(vals_bytes + 64);
        CUDA_OK(cudaMemcpyAsync(L.keys.p, d_keys32, 32ull * n, cudaMemcpyDeviceToDevice, c->st));
        CUDA_OK(cudaMemcpyAsync(L.off.p, d_val_off, 8ull * (n + 1), cudaMemcpyDeviceToDevice, c->st));
        if (vals_bytes) CUDA_OK(cudaMemcpyAsync(L.vals.p, d_vals, vals_bytes, cudaMemcpyDeviceToDevice, c->st));
      }
      trie_root_sorted_dev(c, t.st[0], L.keys.as<uint8_t>(), L.off.as<uint64_t>(), L.vals.as<uint8_t>(), n, t.root, 0, nullptr, true);
      t.n = (uint32_t)n;
    });
  });
}

int ppd_trie_info(const ppd_trie* t, size_t* n_leaves, uint8_t root_out[32]) {
  if (!t) return PPD_ERR_BAD_ARGUMENT;
  if (n_leaves) *n_leaves = t->n;
  if (root_out) memcpy(root_out, t->root, 32);
  return PPD_OK;
}

int ppd_trie_subset_dev(ppd_ctx* c, ppd_trie* t, const uint8_t* d_queries, size_t m, uint8_t** out, size_t* out_len) {
  return guarded(c, [&] {
    stats_reset(c);
    ppd_trie& T = *checked(c, t);
    trie_subset(c, T, handle_query(T, d_queries, m, out, out_len));
  });
}

int ppd_trie_subset(ppd_ctx* c, ppd_trie* t, const uint8_t* queries, size_t m, uint8_t** out, size_t* out_len) {
  return guarded(c, [&] {
    stats_reset(c);
    ppd_trie& T = *checked(c, t);
    SubsetQuery q = handle_query(T, queries, m, out, out_len);
    if (m) {
      c->d_subset[SB_QRAW].reserve((size_t)T.key_len * m);
      CUDA_OK(cudaMemcpyAsync(c->d_subset[SB_QRAW].p, queries, (size_t)T.key_len * m, cudaMemcpyHostToDevice, c->st));
      c->stats.h2d_bytes += (double)((size_t)T.key_len * m);
      q.d_keys = c->d_subset[SB_QRAW].as<uint8_t>();
    }
    trie_subset(c, T, q);
  });
}

int ppd_trie_update_dev(ppd_ctx* c, ppd_trie* t, const uint8_t* d_keys, const uint8_t* d_del, const uint64_t* d_val_off, const uint8_t* d_vals,
                        size_t k, size_t vals_bytes, uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    trie_update(c, *checked(c, t), d_keys, d_del, d_val_off, d_vals, k, vals_bytes, root_out);
  });
}

int ppd_trie_update(ppd_ctx* c, ppd_trie* t, const uint8_t* keys, const uint8_t* del, const uint64_t* val_off, const uint8_t* vals, size_t k,
                    uint8_t root_out[32]) {
  return guarded(c, [&] {
    stats_reset(c);
    ppd_trie& T = *checked(c, t);
    if (k == 0 || k >= 0x7ffffffeull) {
      trie_update(c, T, nullptr, nullptr, nullptr, nullptr, k, 0, root_out);  // nothing to do, or the argument error
      return;
    }
    const size_t vb = val_off[k];
    c->d_keys.reserve((size_t)T.key_len * k);
    c->d_msg_off.reserve(8 * (k + 1));
    c->d_vals.reserve(vb + 64);
    CUDA_OK(cudaMemcpyAsync(c->d_keys.p, keys, (size_t)T.key_len * k, cudaMemcpyHostToDevice, c->st));
    CUDA_OK(cudaMemcpyAsync(c->d_msg_off.p, val_off, 8 * (k + 1), cudaMemcpyHostToDevice, c->st));
    CUDA_OK(cudaMemcpyAsync(c->d_vals.p, vals, vb, cudaMemcpyHostToDevice, c->st));
    size_t up = (size_t)T.key_len * k + 8 * (k + 1) + vb;
    if (del) {
      c->d_msg.reserve(k);
      CUDA_OK(cudaMemcpyAsync(c->d_msg.p, del, k, cudaMemcpyHostToDevice, c->st));
      up += k;
    }
    c->stats.h2d_bytes += (double)up;
    trie_update(c, T, c->d_keys.as<uint8_t>(), del ? c->d_msg.as<uint8_t>() : nullptr, c->d_msg_off.as<uint64_t>(), c->d_vals.as<uint8_t>(), k, vb,
                root_out);
  });
}

void ppd_trie_destroy(ppd_trie* t) {
  if (!t) return;
  ppd_ctx* c = t->ctx;
  cudaSetDevice(c->device);
  c->tries.erase(std::remove(c->tries.begin(), c->tries.end(), t), c->tries.end());
  t->release();
  delete t;
}

}  // extern "C"
