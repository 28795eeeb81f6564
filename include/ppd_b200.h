/* ppd_b200.h — C ABI of libppd_b200.so, the B200 (sm_100a) implementation of
 * proof-protocol-decoder's hot path.
 *
 * The reference has no FFI of its own for this path: its boundary is the Rust
 * method `BlockTrace::into_txn_proof_gen_ir` (protocol_decoder/src/processed_block_trace.rs:38-45).
 * Each entry point below names the reference interface it stands in for; the
 * Rust shim that binds them (extern "C" block + build.rs) is in INTEGRATION.md.
 *
 * Conventions: plain pointers and sizes only; inputs are caller-owned and only
 * borrowed for the call; outputs returned through `uint8_t** out` are allocated
 * by the library and released with ppd_free(); every call returns a ppd_status
 * (include/ppd_status.h) and never unwinds or aborts across the boundary.  A
 * context is bound to one CUDA device and is not thread-safe; use one context
 * per (thread, device).  There is NO CPU fallback: if no CUDA device is usable
 * ppd_ctx_create fails with PPD_ERR_CUDA.
 *
 * Wire formats (FlatBlock, IrDump, PreImageDump): include/ppd_flat.h.
 */
#ifndef PPD_B200_H
#define PPD_B200_H

#include <stddef.h>
#include <stdint.h>

#include "ppd_flat.h"
#include "ppd_status.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ppd_ctx ppd_ctx;

/* Work counters of the last call on a context. */
typedef struct ppd_stats {
  uint64_t nodes_hashed;       /* Keccak invocations over trie-node encodings (HashedPartialTrie::hash work) */
  uint64_t node_permutations;  /* keccak-f[1600] permutations spent on them */
  uint64_t key_hashes;         /* utils::hash calls: addresses, slots, code */
  uint64_t key_permutations;
  uint64_t node_bytes;         /* bytes of RLP absorbed by those invocations */
  uint64_t arena_nodes;        /* node records resident in HBM */
  uint64_t levels;             /* level launches */
  double gpu_ms;               /* device time of the kernels of the call (CUDA events) */
  double h2d_bytes, d2h_bytes;
  uint64_t kernel_launches;
  uint64_t witnesses_on_gpu;      /* compact witnesses whose parse and pre-image arena were built by the GPU (ppd_parse.cu) */
  uint64_t witness_instructions;  /* instructions of those witnesses */
  uint64_t witness_bytes;         /* bytes of those witnesses */
  double parse_gpu_ms;            /* device time of their parse / arena kernels (CUDA events) */
  uint64_t level_launches;        /* launches of the level-hashing kernel (one per level per block) */
  uint64_t marks_on_gpu;          /* create_trie_subset marking walks (one per accessed key per txn) done by the device */
  uint64_t txn_loops_on_gpu;      /* blocks whose txn loop (decoding.rs:80-177: deltas, subsets, roots) ran on the device (ppd_txn.cu) */
  double txn_gpu_ms;              /* device time of those loops (CUDA events) */
  double dump_gpu_ms;             /* device time of the IrDump kernels (ppd_dump.cu) */
  double host_busy_ms;            /* CPU time of the blocks' host threads (thread CPU clock: sleeping for the device does not count), summed over blocks */
  double host_wait_ms;            /* ... and their time waiting for the device */
} ppd_stats;

int ppd_ctx_create(int device, ppd_ctx** out);
void ppd_ctx_destroy(ppd_ctx* ctx);
/* message of the last non-OK status on this context ("" if none).  For the TraceParsingError statuses (21-25,
 * decoding.rs:31-49) the sentence is followed by "; " and the variant's payload as key=value words — hashed_addr=<64 hex>,
 * trie_type=State|Storage|Receipt|Txn, addr=<40 hex> hashed_addr=<64 hex> amount=<64 hex>, bytes=<hex> (csrc/err_detail.h) —
 * from which the shim rebuilds the reference's error value (integration/rust/src/b200/status.rs). */
const char* ppd_last_error(const ppd_ctx* ctx);
void ppd_last_stats(const ppd_ctx* ctx, ppd_stats* out);
void ppd_free(void* p);
/* A page-locked host buffer of n bytes from the library's pool (an ordinary malloc block once the pool's
 * cap is reached); release with ppd_free.  Inputs placed in such a buffer (the Rust shim serialises the
 * BlockTrace of processed_block_trace.rs:38-45 straight into one) are read by the GPU's copy engine
 * directly; any other host pointer is accepted too and staged through page-locked memory by the library. */
void* ppd_alloc_pinned(size_t n);

/* utils::hash (protocol_decoder/src/utils.rs:11-13) over a batch: message i is
 * data[offsets[i] .. offsets[i+1]); out32n receives n x 32 bytes.  Host buffers. */
int ppd_keccak256_batch(ppd_ctx* ctx, const uint8_t* data, const uint64_t* offsets, size_t n, uint8_t* out32n);

/* process_compact_prestate_debug (compact/compact_prestate_processing.rs:1262-1281) plus the root
 * of every resulting trie (HashedPartialTrie::hash): TrieCompact bytes -> PreImageDump. */
int ppd_compact_decode(ppd_ctx* ctx, const uint8_t* witness, size_t len, uint8_t** out, size_t* out_len);

/* A Separate{state: Direct, storage: MultipleTries{Direct}} pre-image (trace_protocol.rs:58-108; the DirectPreImage
 * payload of include/ppd_flat.h) re-spelled as the TrieCompact witness of the same tries, on the host, without a
 * context: what ppd_block_decode does first with a kind-2 FlatBlock (csrc/host_direct.cu; processed_block_trace.rs:
 * 130-168 is the reference side, whose storage half is todo!()).  Accounts whose storage trie is not in the payload
 * appear in the witness with their storage root hashed out.  Structure only, no hashing.  Release with ppd_free.
 * Returns PPD_ERR_BAD_FLAT_INPUT for a malformed payload, PPD_PANIC_PRE_IMAGE_ACCOUNT_DECODE for a state leaf that is
 * not an RLP account. */
int ppd_direct_to_compact(const uint8_t* direct, size_t len, uint8_t** out, size_t* out_len);

/* BlockTrace::into_txn_proof_gen_ir (processed_block_trace.rs:38-50 -> decoding.rs:80-177):
 * FlatBlock -> IrDump (one GenerationInputs per txn, plus dummies / the withdrawal entry). */
int ppd_block_decode(ppd_ctx* ctx, const uint8_t* flat_block, size_t len, uint8_t** out, size_t* out_len);

/* The same over n independent blocks, decoded concurrently (up to 64 resident at a time, each on its own stream and
 * HBM pools; every block's tries are hashed by level-synchronous sweeps of its own).  statuses[i] is the status of
 * block i; outs[i] is NULL for a failed block.  On a non-OK return (a CUDA failure) no output is handed out: every
 * outs[i] is NULL. */
int ppd_blocks_decode_batch(ppd_ctx* ctx, const uint8_t* const* flat_blocks, const size_t* lens, size_t n, uint8_t** outs,
                            size_t* out_lens, int* statuses);

/* The same for a caller that consumes blocks as they finish (a node that keeps feeding blocks: the pipeline never drains
 * between calls' worth of blocks, and only the outputs in flight are held): `done` is called once per block, from one
 * of the library's host threads, as soon as that block is decoded — in completion order, not input order; `out` (NULL
 * for a failed block) is the callee's to release with ppd_free.  Calls of `done` may overlap on different threads.
 * A non-OK return is a CUDA failure; blocks delivered before it stay delivered. */
typedef void (*ppd_block_done_fn)(void* user, size_t index, int status, uint8_t* out, size_t out_len);
int ppd_blocks_decode_stream(ppd_ctx* ctx, const uint8_t* const* flat_blocks, const size_t* lens, size_t n, ppd_block_done_fn done, void* user);

/* Measurement hook: re-run kernels of the last ppd_block_decode / ppd_blocks_decode_batch on what is still resident
 * in HBM (no host work, no copies); returns the device time (CUDA events).  `what` selects the stages, which every
 * lane runs in pipeline order, lanes concurrently: the witness parse + pre-image arena (ppd_parse.cu), key hashing and
 * the level sweeps (ppd_kernels.cu), the txn loop with its join / account table / op sort (ppd_txn.cu), IR sizing and
 * emit (ppd_dump.cu).  TXN and DUMP apply to blocks whose txn loop ran on the device. */
#define PPD_REPLAY_PARSE 1u
#define PPD_REPLAY_HASH 2u
#define PPD_REPLAY_TXN 4u
#define PPD_REPLAY_DUMP 8u
#define PPD_REPLAY_ALL 15u
int ppd_replay_last(ppd_ctx* ctx, unsigned what, double* gpu_ms_out);
/* How many lanes (= blocks) a replay covers: the lanes of the last decode call that still hold a block, at most 30 (every
 * lane replays on a stream of its own, and the device runs 32 streams side by side). */
size_t ppd_replay_lanes(const ppd_ctx* ctx);
/* = ppd_replay_last(ctx, PPD_REPLAY_HASH, ...) */
int ppd_replay_last_hashing(ppd_ctx* ctx, double* gpu_ms_out);
/* = ppd_replay_last(ctx, PPD_REPLAY_PARSE, ...): the compact-witness kernels (instruction boundaries, stack machine, arena emit: the GPU form of
 * compact_prestate_processing.rs:683-875, 325-668 and compact_to_partial_trie.rs:37-165) of the last call. */
int ppd_replay_last_parse(ppd_ctx* ctx, double* gpu_ms_out);

/* Measurement hook: ceilings of the Keccak roofline (csrc/ppd_microbench.cu).  variant 0: issue rate of
 * dependent-free LOP3/SHF (units = ALU instructions); variants 1..: keccak-f[1600] on a register-resident
 * state with different unroll factors / ALU-vs-FMA-pipe rotation splits (units = permutations). */
int ppd_microbench(ppd_ctx* ctx, int variant, uint32_t blocks_per_sm, uint32_t iters, double* gpu_ms_out, double* units_out,
                   uint32_t* digest_out);

/* HashedPartialTrie::hash of the trie holding n leaves with 32-byte keys, given sorted by key
 * (the state-trie rehash of config 5).  value i = vals[val_off[i] .. val_off[i+1]) is stored as
 * given (it is the already-RLP-encoded leaf payload).  Host buffers. */
int ppd_trie_root_sorted_leaves(ppd_ctx* ctx, const uint8_t* keys32, const uint64_t* val_off, const uint8_t* vals, size_t n,
                                uint8_t root_out[32]);

/* Device-resident variant for measurement: pointers are DEVICE pointers (cudaMalloc'ed by the
 * caller, e.g. torch tensors); only the 32-byte root is copied back. */
int ppd_trie_root_sorted_leaves_dev(ppd_ctx* ctx, const uint8_t* d_keys32, const uint64_t* d_val_off, const uint8_t* d_vals,
                                    size_t n, size_t vals_bytes, uint8_t root_out[32]);

#define PPD_LEAVES_HASH_KEYS 1u /* key i is keccak256(keys[i*key_len .. +key_len)), not the bytes themselves */
/* HashedPartialTrie::hash() of the trie obtained by inserting (key_0, val_0) ... (key_{n-1}, val_{n-1}) in this order
 * into an empty trie (eth_trie_utils `insert`, compact_to_partial_trie.rs:105,125): any key order, and a repeated key
 * keeps the value of its LAST occurrence.  Without PPD_LEAVES_HASH_KEYS key_len must be 32; with it, 1 <= key_len <= 135
 * (20: addresses, 32: slots).  Values as for ppd_trie_root_sorted_leaves (already-RLP-encoded payloads, taken as given).
 * Inputs are only read, never reordered in place.  Never returns PPD_ERR_UNSORTED_KEYS.  PPD_ERR_BAD_ARGUMENT for unknown
 * flag bits, a bad key_len, n >= 2^31 - 2, or val_off decreasing anywhere or ending past vals_bytes.  The leaves are
 * sorted, de-duplicated and gathered on the GPU (csrc/ppd_leaves.cu), then built as by the sorted entry.
 * DEVICE pointers, complete when the call is made (the library reads them on a stream of its own); vals_bytes =
 * readable bytes of d_vals. */
int ppd_trie_root_leaves_dev(ppd_ctx* ctx, const uint8_t* d_keys, uint32_t key_len, uint32_t flags, const uint64_t* d_val_off,
                             const uint8_t* d_vals, size_t n, size_t vals_bytes, uint8_t root_out[32]);
/* The same from host buffers. */
int ppd_trie_root_leaves(ppd_ctx* ctx, const uint8_t* keys, uint32_t key_len, uint32_t flags, const uint64_t* val_off,
                         const uint8_t* vals, size_t n, uint8_t root_out[32]);

/* create_trie_subset (decoding.rs:551-602, eth_trie_utils trie_subsets.rs) of the trie over the leaves, for the m query
 * keys: the minimal sub-trie that holds the path to every query key, each node off those paths replaced by HASH(its
 * hash), or kept whole when it encodes to fewer than 32 bytes.  The form a pre-image takes (the Direct state trie of a
 * DirectPreImage, every trie of a GenerationInputs), cut on the GPU from the trie the root entries build.
 * The trie and the leaves follow the matching root entry exactly (insertion order, the last value wins,
 * PPD_LEAVES_HASH_KEYS, the same argument checks; the sorted entry returns PPD_ERR_UNSORTED_KEYS unless the keys are
 * strictly ascending).  Queries: m keys of key_len bytes, keccak256-hashed first under PPD_LEAVES_HASH_KEYS like the
 * leaf keys, otherwise 32 bytes; any order, repeats allowed.  A key absent from the trie keeps the path down to where it
 * leaves the trie (a branch with an empty slot, an extension whose nibbles differ, a leaf with another suffix): the
 * proof of its absence.  m = 0 gives the untouched root, HASH(root) (the root of a trie of 32-byte keys always
 * encodes to 32 bytes or more).  m >= 2^31 - 2 returns PPD_ERR_BAD_ARGUMENT.
 * *out: one Trie in the pre-order Node form of ppd_flat.h (no header), leaves holding the value bytes as given; the
 * empty trie gives a single PPD_NODE_EMPTY.  Release with ppd_free.  root_out: the root of the whole trie, which is also
 * the hash of the subset.  The subset is marked, sized and written on the GPU (csrc/ppd_subset.cu) over the builder's
 * arrays within the same call; ppd_last_stats counts its kernels in gpu_ms and kernel_launches, its copies in d2h_bytes.
 * DEVICE pointers (keys, offsets, values and queries), complete when the call is made. */
int ppd_trie_subset_leaves_dev(ppd_ctx* ctx, const uint8_t* d_keys, uint32_t key_len, uint32_t flags, const uint64_t* d_val_off,
                               const uint8_t* d_vals, size_t n, size_t vals_bytes, const uint8_t* d_queries, size_t m,
                               uint8_t** out, size_t* out_len, uint8_t root_out[32]);
/* The same from host buffers. */
int ppd_trie_subset_leaves(ppd_ctx* ctx, const uint8_t* keys, uint32_t key_len, uint32_t flags, const uint64_t* val_off,
                           const uint8_t* vals, size_t n, const uint8_t* queries, size_t m,
                           uint8_t** out, size_t* out_len, uint8_t root_out[32]);
/* The same over leaves sorted by 32-byte key (ppd_trie_root_sorted_leaves_dev: no sort), with 32-byte queries.  DEVICE
 * pointers. */
int ppd_trie_subset_sorted_leaves_dev(ppd_ctx* ctx, const uint8_t* d_keys32, const uint64_t* d_val_off, const uint8_t* d_vals,
                                      size_t n, size_t vals_bytes, const uint8_t* d_queries32, size_t m,
                                      uint8_t** out, size_t* out_len, uint8_t root_out[32]);

/* A trie kept resident in HBM: built once from leaves, then cut into subsets and updated in place, each update
 * re-hashing only the nodes on the paths of the keys it writes or deletes (csrc/gpu_trie.cu, csrc/ppd_update.cu).
 * A handle fixes its key_len and PPD_LEAVES_HASH_KEYS when it is created; queries and update keys take the same length
 * and are hashed the same way (the sorted create: 32-byte keys, no hashing).  A handle belongs to its context, which
 * stays not thread-safe; other calls on the context (one-shot entries, block decodes, other handles) may come between
 * handle calls and do not disturb it.  ppd_ctx_destroy releases every handle still alive.  A call that returns an
 * error leaves the handle's leaves, root and subsets as they were (an out-of-memory PPD_ERR_CUDA included).  A NULL
 * handle, or one passed with another context than the one that created it, is PPD_ERR_BAD_ARGUMENT. */
typedef struct ppd_trie ppd_trie;
/* Build and keep: the trie, contract and argument checks of the matching root entry (the any-order leaf entries, or
 * the sorted device entry); root_out as they give it.  *out: the new handle.  Inputs are only borrowed for the call:
 * the sorted create copies vals_bytes bytes of values, so it also returns PPD_ERR_BAD_ARGUMENT when val_off decreases
 * or val_off[n] exceeds vals_bytes.  Device keys, queries and values may sit at any alignment. */
int ppd_trie_create_leaves_dev(ppd_ctx* ctx, const uint8_t* d_keys, uint32_t key_len, uint32_t flags, const uint64_t* d_val_off,
                               const uint8_t* d_vals, size_t n, size_t vals_bytes, ppd_trie** out, uint8_t root_out[32]);
int ppd_trie_create_leaves(ppd_ctx* ctx, const uint8_t* keys, uint32_t key_len, uint32_t flags, const uint64_t* val_off,
                           const uint8_t* vals, size_t n, ppd_trie** out, uint8_t root_out[32]);
int ppd_trie_create_sorted_leaves_dev(ppd_ctx* ctx, const uint8_t* d_keys32, const uint64_t* d_val_off, const uint8_t* d_vals,
                                      size_t n, size_t vals_bytes, ppd_trie** out, uint8_t root_out[32]);
/* The current leaf count and root, from the host (no device work). */
int ppd_trie_info(const ppd_trie* t, size_t* n_leaves, uint8_t root_out[32]);
/* create_trie_subset of the current trie for m query keys; the output as the subset leaf entries give it.  Nothing is
 * rebuilt.  DEVICE queries, or host queries. */
int ppd_trie_subset_dev(ppd_ctx* ctx, ppd_trie* t, const uint8_t* d_queries, size_t m, uint8_t** out, size_t* out_len);
int ppd_trie_subset(ppd_ctx* ctx, ppd_trie* t, const uint8_t* queries, size_t m, uint8_t** out, size_t* out_len);
/* Applies k updates in input order: update i writes (key_i, vals[val_off[i] .. val_off[i + 1])), or deletes key_i when
 * del is non-NULL and del[i] != 0 (a delete ignores its value range).  The result is that of eth_trie_utils `insert` /
 * `delete` applied in this order: the last update of a key wins, deleting an absent key changes nothing, deleting every
 * key gives EMPTY_TRIE_HASH.  k = 0 changes nothing and hashes nothing.  Arguments are checked as the leaf entries check
 * them (val_off on the device, k >= 2^31 - 2 rejected), and an update that would leave 2^31 - 2 or more leaves is
 * PPD_ERR_BAD_ARGUMENT.  root_out: the new root.  ppd_last_stats: gpu_ms covers the whole call, nodes_hashed counts the
 * nodes the update re-hashed.  DEVICE pointers (keys, del, val_off, vals; vals_bytes = readable bytes of d_vals), or
 * host buffers. */
int ppd_trie_update_dev(ppd_ctx* ctx, ppd_trie* t, const uint8_t* d_keys, const uint8_t* d_del, const uint64_t* d_val_off,
                        const uint8_t* d_vals, size_t k, size_t vals_bytes, uint8_t root_out[32]);
int ppd_trie_update(ppd_ctx* ctx, ppd_trie* t, const uint8_t* keys, const uint8_t* del, const uint64_t* val_off,
                    const uint8_t* vals, size_t k, uint8_t root_out[32]);
/* Releases the handle and its device memory (NULL: no-op). */
void ppd_trie_destroy(ppd_trie* t);

/* One huge trie over several streams or GPUs (SURVEY.md 8e (3)): the leaves are split by their first `base_depth`
 * nibbles; each part is hashed like a whole trie, except that its nodes sit `base_depth` nibbles below the root
 * (ref_out = the hash of the part's top node, the 32 bytes the node above embeds).  Every key of the part must share
 * those nibbles, and the top node must encode to at least 32 bytes, or the node above would embed its raw encoding
 * instead: either violation returns PPD_ERR_BAD_ARGUMENT.  Short tops exist from base_depth 9 on (one leaf with a
 * one-byte value encodes to 31 bytes there); base_depth 1 always gives 32 bytes or more.  DEVICE pointers. */
int ppd_trie_subroot_sorted_leaves_dev(ppd_ctx* ctx, const uint8_t* d_keys32, const uint64_t* d_val_off, const uint8_t* d_vals, size_t n,
                                       size_t vals_bytes, uint32_t base_depth, uint8_t ref_out[32]);
/* ... and the branch over them: child_hashes16x32[i] is the ref of the part whose next nibble is i (used when bit i of
 * `mask` is set); root_out = HashedPartialTrie::hash() of that branch.  Host buffers; hashed on the GPU. */
int ppd_trie_root_from_children(ppd_ctx* ctx, const uint8_t* child_hashes16x32, uint32_t mask, uint8_t root_out[32]);

#ifdef __cplusplus
}
#endif
#endif
