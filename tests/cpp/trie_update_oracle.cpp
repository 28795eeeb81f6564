// trie_update_oracle.cpp — the CPU oracle's insert / delete (oracle/ppd_oracle.cpp, eth_trie_utils trie_ops.rs) applied to
// a trie built from leaves, for tests/test_trie_handle.py.  Test infrastructure: compiled by that test into a temporary
// shared library, including the oracle's own code unchanged.
#include "../../oracle/ppd_oracle.cpp"

extern "C" {

// The trie of the n leaves (inserted in input order), then the k updates in order: update i deletes ukeys32[i] when
// del[i] != 0, else inserts (ukeys32[i], uvals[uoff[i] .. uoff[i + 1])).  root_out: its hash.  When out is non-NULL,
// create_trie_subset of the result for m 32-byte queries, in the pre-order Node form (include/ppd_flat.h).
int oracle_trie_update(const uint8_t* keys32, const uint64_t* val_off, const uint8_t* vals, size_t n, const uint8_t* ukeys32, const uint8_t* del,
                       const uint64_t* uoff, const uint8_t* uvals, size_t k, const uint8_t* queries32, size_t m, uint8_t* root_out, uint8_t** out,
                       size_t* out_len, char* err, size_t err_cap) {
  return guarded(
      [&] {
        NodeP t = EMPTY_NODE;
        for (size_t i = 0; i < n; i++)
          t = trie_insert(t, nibs_from_bytes(keys32 + 32 * i, 32), InsertVal{false, Bytes(vals + val_off[i], vals + val_off[i + 1]), {}});
        for (size_t i = 0; i < k; i++) {
          Nibs key = nibs_from_bytes(ukeys32 + 32 * i, 32);
          if (del[i]) {
            NodeP d = trie_delete(t, key);
            if (d) t = d;  // nullptr: the key is absent, the trie unchanged
          } else
            t = trie_insert(t, key, InsertVal{false, Bytes(uvals + uoff[i], uvals + uoff[i + 1]), {}});
        }
        const H256 h = trie_hash(t);
        memcpy(root_out, h.b, 32);
        if (!out) return 0;
        std::vector<Nibs> qs;
        for (size_t i = 0; i < m; i++) qs.push_back(nibs_from_bytes(queries32 + 32 * i, 32));
        Writer w;
        dump_node(w, *create_trie_subset(t, qs));
        return finish(w.b, out, out_len);
      },
      err, err_cap);
}

}  // extern "C"
