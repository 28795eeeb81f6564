// trie_subset_oracle.cpp — the CPU oracle's create_trie_subset (oracle/ppd_oracle.cpp, eth_trie_utils trie_subsets.rs)
// over a trie built from leaves, for tests/test_trie_subset.py.  Test infrastructure: compiled by that test into a
// temporary shared library next to the oracle's own code, which it includes unchanged.
#include "../../oracle/ppd_oracle.cpp"

extern "C" {

// create_trie_subset of the trie oracle_trie_root_from_leaves builds (the leaves inserted in input order), for m
// 32-byte query keys, written as one Trie in the pre-order Node form (include/ppd_flat.h).
int oracle_trie_subset_from_leaves(const uint8_t* keys32, const uint64_t* val_off, const uint8_t* vals, size_t n, const uint8_t* queries32, size_t m,
                                   uint8_t** out, size_t* out_len, char* err, size_t err_cap) {
  return guarded(
      [&] {
        NodeP t = EMPTY_NODE;
        for (size_t i = 0; i < n; i++) {
          Nibs k = nibs_from_bytes(keys32 + 32 * i, 32);
          t = trie_insert(t, k, InsertVal{false, Bytes(vals + val_off[i], vals + val_off[i + 1]), {}});
        }
        std::vector<Nibs> keys;
        for (size_t i = 0; i < m; i++) keys.push_back(nibs_from_bytes(queries32 + 32 * i, 32));
        Writer w;
        dump_node(w, *create_trie_subset(t, keys));
        return finish(w.b, out, out_len);
      },
      err, err_cap);
}

}  // extern "C"
