// host_direct.cu — Separate{state: Direct, storage: MultipleTries{Direct}} pre-images (FlatBlock pre_image_kind 2).
//
// Reference: BlockTraceTriePreImages::Separate (trace_protocol.rs:58-108) -> process_separate_trie_pre_images
// (processed_block_trace.rs:130-168).  There the state trie of a Direct pre-image is taken as it is (`t.0`, :145)
// and extra_code_hash_mappings is None (:139); process_multiple_storage_tries is todo!() (:164-168).  Kind 2 completes
// it the way process_state_trie is written: every entry of the map is the trie it holds, keyed by hashed address.
//
// A direct pre-image is the SAME tree the compact witness spells in post-order, so the host re-spells it: one pass
// over the pre-order Node form (include/ppd_flat.h) writes the witness opcodes of compact_prestate_processing.rs:744-875
// -- a hashed-out node as HASH, a branch as its children then BRANCH(mask), an account leaf as [HASH(code hash)] [its
// storage trie | HASH(storage root)] ACCOUNT_LEAF(key, flags, nonce, balance) -- and the block then takes the witness
// path: GPU parse, GPU hashing, the device txn loop, GPU IR dump.  Structure only: no hashing here.  The witness is
// written into a caller-owned buffer (page-locked for a decode: the copy engine reads it as it is).
//
// What differs from a Combined pre-image is WHICH accounts have a storage trie: by hashed address as given, not by
// root hash (compact_to_partial_trie.rs:167-190).  `direct_keep` records the addresses of the map.  The device txn loop
// joins accounts to tries by these addresses (ppd_txn.cu: join_addr_*_kernel); the host path drops every other entry
// after the pre-image is built (direct_filter_storage) and skips the by-root join.
//
// Preconditions (a pre-image a tracer would send meets them; an input that does not is rejected with
// PPD_ERR_BAD_FLAT_INPUT, or noted): every state leaf is an RLP account (else PPD_PANIC_PRE_IMAGE_ACCOUNT_DECODE, as
// when the reference first decodes it); nonces fit 64 bits; storage leaves hold one RLP string; branches carry no
// value; every storage trie belongs to an account of the state trie; an account's storage_root field is the root of
// the trie sent for it (the witness path derives the field from the trie).  A trie that is not the canonical trie
// of its items is rebuilt from its items, as for a witness.
#include "host_pipeline.h"

namespace ppd {

namespace {

struct DirectEncoder {
  FlatReader r;
  PVec<uint8_t>& out;
  std::unordered_map<H256, std::pair<size_t, bool>, H256Hasher> storage_at;  // hashed address -> (offset of its trie, used)
  uint8_t path[160];

  [[noreturn]] void bad(const char* why) { throw Fail{PPD_ERR_BAD_FLAT_INPUT, std::string("direct pre-image: ") + why}; }

  void cbor_head(uint32_t major, uint64_t v) {
    const uint8_t m = (uint8_t)(major << 5);
    if (v < 24) {
      out.push_back(m | (uint8_t)v);
      return;
    }
    const int width = v < 0x100 ? 1 : v < 0x10000 ? 2 : v < 0x100000000ull ? 4 : 8;
    out.push_back(m | (uint8_t)(width == 1 ? 24 : width == 2 ? 25 : width == 4 ? 26 : 27));
    for (int k = width - 1; k >= 0; k--) out.push_back((uint8_t)(v >> (8 * k)));
  }
  void cbor_bytes(const uint8_t* p, size_t n) {
    cbor_head(2, n);
    out.append(p, n);
  }
  // the inverse of key_bytes_to_nibbles (compact_prestate_processing.rs:1338-1390): a flag byte (bit 0: odd count), then
  // the nibbles packed high first
  void compact_key(const uint8_t* nib, uint32_t cnt) {
    if (cnt == 0) {
      cbor_head(2, 0);
      return;
    }
    uint8_t buf[34];
    buf[0] = (uint8_t)(cnt & 1);
    const uint32_t nb = (cnt + 1) / 2;
    for (uint32_t k = 0; k < nb; k++) buf[1 + k] = (uint8_t)((nib[2 * k] << 4) | (2 * k + 1 < cnt ? nib[2 * k + 1] : 0));
    cbor_bytes(buf, 1 + nb);
  }
  uint32_t read_nibbles(uint8_t* dst, uint32_t depth) {
    const uint32_t cnt = r.u8();
    if (cnt > 64 || depth + cnt > 64) bad("key longer than 64 nibbles");
    const uint8_t* p = r.raw(cnt);
    for (uint32_t k = 0; k < cnt; k++) {
      if (p[k] > 15) bad("nibble above 15");
      dst[k] = p[k];
    }
    return cnt;
  }
  // moves the reader past one node
  void skip(int guard) {
    if (guard > 140) bad("nested deeper than any 64-nibble key allows");
    switch (r.u8()) {
      case PPD_NODE_EMPTY:
        return;
      case PPD_NODE_HASH:
        r.raw(32);
        return;
      case PPD_NODE_BRANCH:
        for (int k = 0; k < 16; k++) skip(guard + 1);
        r.bytes();
        return;
      case PPD_NODE_EXTENSION:
        r.raw(r.u8());
        skip(guard + 1);
        return;
      case PPD_NODE_LEAF:
        r.raw(r.u8());
        r.bytes();
        return;
      default:
        bad("unknown node kind");
    }
  }
  // one node of a trie, its subtree first; false: the node is Empty (nothing written)
  bool node(uint32_t depth, bool is_state, bool is_root) {
    const uint8_t kind = r.u8();
    switch (kind) {
      case PPD_NODE_EMPTY:
        if (is_root) out.push_back(PPD_OP_EMPTY_ROOT);
        return is_root;
      case PPD_NODE_HASH: {
        const uint8_t* h = r.raw(32);
        out.push_back(PPD_OP_HASH);
        out.append(h, 32);
        return true;
      }
      case PPD_NODE_BRANCH: {
        if (depth >= 64) bad("branch below 64 nibbles");
        uint32_t mask = 0;
        for (uint32_t k = 0; k < 16; k++) {
          path[depth] = (uint8_t)k;
          if (node(depth + 1, is_state, false)) mask |= 1u << k;
        }
        if (r.bytes().n) bad("a branch with a value");
        if (!mask) bad("a branch without children");
        out.push_back(PPD_OP_BRANCH);
        cbor_head(0, mask);
        return true;
      }
      case PPD_NODE_EXTENSION: {
        const uint32_t cnt = read_nibbles(path + depth, depth);
        if (!node(depth + cnt, is_state, false)) bad("an extension over an empty node");
        out.push_back(PPD_OP_EXTENSION);
        compact_key(path + depth, cnt);
        return true;
      }
      case PPD_NODE_LEAF: {
        const uint32_t cnt = read_nibbles(path + depth, depth);
        const Span v = r.bytes();
        if (is_state)
          account_leaf(depth, cnt, v);
        else
          value_leaf(depth, cnt, v);
        return true;
      }
      default:
        bad("unknown node kind");
    }
  }
  void value_leaf(uint32_t depth, uint32_t cnt, Span v) {
    // the witness carries the slot value, the trie its RLP string (compact_to_partial_trie.rs:119)
    RlpItem it;
    if (!rlp_item(v.p, v.n, it) || it.is_list || it.total_len != v.n) bad("a storage leaf that is not one RLP string");
    out.push_back(PPD_OP_LEAF);
    compact_key(path + depth, cnt);
    cbor_bytes(it.payload, it.payload_len);
  }
  void account_leaf(uint32_t depth, uint32_t cnt, Span v) {
    // AccountRlp {nonce, balance, storage_root, code_hash} (compact_to_partial_trie.rs:141-165 builds it; here it is read)
    RlpItem top, f[4];
    if (!rlp_item(v.p, v.n, top) || !top.is_list) fail(PPD_PANIC_PRE_IMAGE_ACCOUNT_DECODE, "state leaf is not an account");
    const uint8_t* q = top.payload;
    size_t m = top.payload_len;
    for (int k = 0; k < 4; k++) {
      if (!rlp_item(q, m, f[k]) || f[k].is_list) fail(PPD_PANIC_PRE_IMAGE_ACCOUNT_DECODE, "state leaf is not an account");
      q += f[k].total_len, m -= f[k].total_len;
    }
    if (f[0].payload_len > 32 || f[1].payload_len > 32 || (f[0].payload_len && f[0].payload[0] == 0) || (f[1].payload_len && f[1].payload[0] == 0) ||
        f[2].payload_len != 32 || f[3].payload_len != 32)
      fail(PPD_PANIC_PRE_IMAGE_ACCOUNT_DECODE, "state leaf is not an account");
    if (f[0].payload_len > 8) bad("an account nonce wider than 64 bits");
    uint64_t nonce = 0;
    for (size_t k = 0; k < f[0].payload_len; k++) nonce = (nonce << 8) | f[0].payload[k];
    // hashed address: the leaf's full key, right-aligned (utils.rs:49-59)
    const uint32_t klen = depth + cnt;
    H256 haddr;
    memset(haddr.b, 0, 32);
    for (uint32_t k = 0; k < klen; k++) {
      const uint32_t posn = 64 - klen + k;
      haddr.b[posn >> 1] |= (uint8_t)((posn & 1) ? path[k] : (path[k] << 4));
    }
    uint8_t flags = 0;
    if (memcmp(f[3].payload, EMPTY_CODE_HASH, 32) != 0) {
      flags |= 1;
      out.push_back(PPD_OP_HASH);
      out.append(f[3].payload, 32);
    }
    auto s = storage_at.find(haddr);
    if (s != storage_at.end()) {
      if (s->second.second) bad("two state leaves with one hashed address");
      s->second.second = true;
      flags |= 2;
      // the account's own storage trie, spelled in place (the state trie's reader position and path are kept)
      const size_t keep_pos = r.pos;
      uint8_t keep_path[64];
      memcpy(keep_path, path, 64);
      r.pos = s->second.first;
      node(0, false, true);
      r.pos = keep_pos;
      memcpy(path, keep_path, 64);
    } else if (memcmp(f[2].payload, EMPTY_TRIE_HASH, 32) != 0) {
      flags |= 2;  // storage that was not sent: the root alone
      out.push_back(PPD_OP_HASH);
      out.append(f[2].payload, 32);
    }
    if (nonce) flags |= 4;
    if (f[1].payload_len) flags |= 8;
    out.push_back(PPD_OP_ACCOUNT_LEAF);
    compact_key(path + depth, cnt);
    out.push_back(flags);
    if (flags & 4) cbor_head(0, nonce);
    if (flags & 8) cbor_bytes(f[1].payload, f[1].payload_len);
    if (flags & 1) cbor_head(0, 0);  // code size: read and dropped by the parser
  }
};

}  // namespace

void direct_to_compact(BlockJob& b, PVec<uint8_t>& wit) {
  wit.clear();
  wit.reserve((size_t)b.direct.n + (size_t)b.direct.n / 8 + 64);
  DirectEncoder e{FlatReader{b.direct.p, b.direct.n}, wit, {}, {}};
  // where every storage trie starts
  e.skip(0);
  const uint32_t ns = e.r.u32();
  if ((uint64_t)ns * 33 > e.r.n - e.r.pos) e.bad("storage trie count exceeds the input");
  e.storage_at.reserve(ns);
  b.direct_keep.clear();
  b.direct_keep.reserve(ns);
  for (uint32_t i = 0; i < ns; i++) {
    H256 h;
    memcpy(h.b, e.r.raw(32), 32);
    if (!e.storage_at.insert({h, {e.r.pos, false}}).second) e.bad("two storage tries for one hashed address");
    b.direct_keep.push_back(h);
    e.skip(0);
  }
  if (e.r.pos != e.r.n) e.bad("bytes after the last storage trie");
  // the witness: header (version 1), then the state trie in post-order
  e.out.push_back(1);
  e.r.pos = 0;
  e.node(0, true, true);
  for (const auto& s : e.storage_at)
    if (!s.second.second) e.bad("a storage trie for an account the state trie does not hold");
  if (e.out.size() >= 0xfff00000ull) e.bad("too large");
  const size_t n = e.out.size();
  e.out.resize(n + 64);
  memset(e.out.data() + n, 0, 64);  // readable past the end, like every witness buffer
  b.compact = Span{e.out.data(), (uint32_t)n};
}

// after the pre-image is built: the accounts that have a storage trie are those of the map (by hashed address)
void direct_filter_storage(BlockJob& b) {
  std::unordered_set<H256, H256Hasher> keep(b.direct_keep.begin(), b.direct_keep.end());
  for (const BlockJob::PreAccount& pa : b.pre_accounts)
    if (!keep.count(pa.haddr)) b.storage.erase(pa.haddr);
}

}  // namespace ppd

extern "C" int ppd_direct_to_compact(const uint8_t* direct, size_t len, uint8_t** out, size_t* out_len) {
  if (!out || !out_len || (!direct && len)) return PPD_ERR_BAD_ARGUMENT;
  *out = nullptr, *out_len = 0;
  if (len > 0xfff00000ull) return PPD_ERR_BAD_FLAT_INPUT;
  try {
    ppd::BlockJob b;
    ppd::PVec<uint8_t> wit;
    b.direct = ppd::Span{direct, (uint32_t)len};
    ppd::direct_to_compact(b, wit);
    uint8_t* p = (uint8_t*)malloc(b.compact.n ? b.compact.n : 1);
    if (!p) return PPD_ERR_BAD_ARGUMENT;
    memcpy(p, b.compact.p, b.compact.n);
    *out = p, *out_len = b.compact.n;
    return PPD_OK;
  } catch (const ppd::Fail& e) {
    return e.code;
  } catch (const std::exception&) {
    return PPD_ERR_BAD_FLAT_INPUT;
  }
}
