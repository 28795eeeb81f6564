// ppd_kernels.h — launchers of the sm_100a kernels (ppd_kernels.cu, ppd_build.cu)
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "arena.h"
#include "txn_core.h"

namespace ppd {

void launch_keccak256_batch(const uint8_t* data, const uint64_t* offsets, uint32_t n, uint8_t* out, cudaStream_t st);
void launch_keccak256_ranges(const uint8_t* data, const uint64_t* begin_end, uint32_t n, uint8_t* out, cudaStream_t st);
void launch_hash_level(const ArenaView& A, const uint32_t* order, uint32_t begin, uint32_t end, cudaStream_t st);
// order[] = node ids counting-sorted by (level, class) on the device; n_bins = 64 * levels (<= 4096), bins zeroed by the caller
static const uint32_t ORDER_MAX_BINS = 4096;
// sorts the nodes first .. first + n (n clipped to *n_dev - first when n_dev, a device pointer, is given)
void launch_order_by_level_class(const NodeRec* nodes, const uint16_t* level, uint32_t n, uint32_t n_bins, uint16_t* keys, uint32_t* bins,
                                 uint32_t* order, cudaStream_t st, uint32_t first = 0, const uint32_t* n_dev = nullptr);

// Small and medium copies done by a kernel instead of the copy engines: either side may be page-locked host memory
// (device-accessible under unified addressing).  A copy engine serves its queue in order, so a few words a lane's host
// thread waits for would sit behind every bulk upload / download other lanes have queued; a kernel is not queued there.
struct CopyBatch {
  static const uint32_t MAX = 16;
  void* dst[MAX];
  const void* src[MAX];
  unsigned long long bytes[MAX];
  uint32_t n = 0;
};
void launch_copy_segments(const CopyBatch& B, cudaStream_t st);
void launch_store_u32x2(uint32_t* dst, uint32_t a, uint32_t b, cudaStream_t st);

// ---- ppd_build.cu: trie construction from sorted leaves ----
struct Pyramid {
  const int8_t *L, *m1, *m2, *m3;
};

// bits of the builder's flags word: checked by the host after the LCP pass (the first two) and after hashing (the last)
enum : uint32_t {
  BUILD_F_UNSORTED = 1,   // keys not strictly ascending
  BUILD_F_PREFIX = 2,     // sub-trie: two adjacent keys share fewer than base_depth nibbles
  BUILD_F_SHORT_TOP = 4,  // sub-trie: the top node encodes to fewer than 32 bytes (the parent embeds it, not its hash)
};

struct BuildView {
  const uint8_t* keys;       // [N][32]
  const uint64_t* val_off;   // [N+1]
  const uint8_t* vals;
  uint32_t n;
  int base_depth;            // nibbles every key shares with the trie above (0: a whole trie; the node found is the root)
  Pyramid P;
  const uint32_t* leader;    // [N+1]
  const uint32_t* bidx;      // [N+1] exclusive scan of leader flags
  // branches
  uint8_t* depth;            // [B]
  uint8_t* ext_start;        // [B]  first nibble of the extension above the branch (== depth when none)
  uint32_t* rep;             // [B]  an item below the branch
  uint32_t* child;           // [B][16]
  uint32_t* root_id;         // id of the root node (leaf or branch)
  uint32_t* flags;           // BUILD_F_* (atomicOr)
  // results
  uint8_t* ref;              // [N + B][32]
  uint8_t* ref_len;          // [N + B]
  uint8_t* root_out;         // [32]
  unsigned long long* counters;
};

size_t scan_tmp_words(size_t n);
void exclusive_scan_u32(const uint32_t* in, uint32_t* out, uint32_t n, uint32_t* tmp, cudaStream_t st);
void launch_lcp(const uint8_t* keys, uint32_t n, int8_t* L, uint32_t* flags, cudaStream_t st, int base_depth = 0);
void launch_min64(const int8_t* in, uint32_t n_in, int8_t* out, uint32_t n_out, cudaStream_t st);
void launch_leaders(const int8_t* L, const int8_t* m1, const int8_t* m2, const int8_t* m3, uint32_t n, uint32_t* link_a, uint32_t* link_b,
                    uint32_t* flag, cudaStream_t st);
void launch_branch_info(const BuildView& V, cudaStream_t st);
void launch_child_count(const uint32_t* leader, const uint32_t* bidx, uint32_t n, uint32_t* nchild, cudaStream_t st);
void launch_depth_hist(const uint8_t* depth, const uint32_t* nchild, uint32_t nb, uint32_t* hist, cudaStream_t st);
void launch_branch_scatter(const uint8_t* depth, const uint32_t* nchild, uint32_t nb, uint32_t* cursor, uint32_t* order, cudaStream_t st);
void launch_hash_sorted_leaves(const BuildView& V, cudaStream_t st);
void launch_hash_branch_level(const BuildView& V, const uint32_t* order, uint32_t begin, uint32_t end, cudaStream_t st);

// ---- ppd_leaves.cu: leaves in any order -> the strictly ascending, de-duplicated leaves of the builder ----
uint32_t scan_launches(size_t n);  // kernels launched by exclusive_scan_u32 over n elements
// tmp: at least scan_tmp_words(n) uint64 (exclusive_scan_u64 returns the number of kernels launched)
uint32_t exclusive_scan_u64(const uint64_t* in, uint64_t* out, uint32_t n, uint64_t* tmp, cudaStream_t st);
void launch_check_offsets(const uint64_t* val_off, uint32_t n, uint64_t vals_bytes, uint32_t* flag, cudaStream_t st);
void launch_hash_fixed_keys(const uint8_t* keys, uint32_t key_len, uint32_t n, uint8_t* out32, cudaStream_t st);
void launch_key_word(const uint8_t* keys32, uint32_t n, int w, uint64_t* out_key, uint32_t* out_val, cudaStream_t st);
void launch_digit_counts(const uint64_t* keys, uint32_t n, uint32_t* counts, cudaStream_t st);  // counts[8 * 256], zeroed by the caller
size_t radix_hist_words(uint32_t n);
// one stable pass on byte digit `digit`; hist and hist_scan hold radix_hist_words(n) words, scan_tmp scan_tmp_words(of that)
uint32_t launch_radix_pass(const uint64_t* keys_in, const uint32_t* vals_in, uint64_t* keys_out, uint32_t* vals_out, uint32_t n, int digit,
                           uint32_t* hist, uint32_t* hist_scan, uint32_t* scan_tmp, cudaStream_t st);
void launch_tie_flags(const uint64_t* sorted_keys, uint32_t n, uint32_t* tie, uint32_t* count, cudaStream_t st);
struct TieRuns {
  uint32_t *member, *mpos, *start, *spos;  // [n + 1]: in a tied run / its first element, and their exclusive scans
  uint32_t *cpos, *cidx, *crun;            // per member, compacted: position, input index, run
  uint64_t* cword;                         // ... and the key word being sorted
};
void launch_tie_members(const uint32_t* tie, uint32_t n, uint32_t* member, uint32_t* start, cudaStream_t st);
void launch_tie_compact(const TieRuns& R, const uint8_t* keys32, const uint32_t* idx, uint32_t n, int w, uint64_t* key, uint32_t* val, cudaStream_t st);
void launch_tie_run_key(const TieRuns& R, const uint32_t* order, uint32_t m, uint64_t* key, uint32_t* val, cudaStream_t st);
void launch_tie_writeback(const TieRuns& R, const uint32_t* order, uint32_t m, uint32_t* idx, uint32_t* tie, uint32_t* count, cudaStream_t st);
void launch_keep_last(const uint32_t* tie, const uint32_t* idx, const uint64_t* val_off, uint32_t n, uint32_t* keep, uint64_t* len, cudaStream_t st);
void launch_gather_leaves(const uint8_t* keys32, const uint32_t* idx, const uint64_t* val_off, const uint8_t* vals, uint32_t n, const uint32_t* keep,
                          const uint32_t* kpos, const uint64_t* koff, uint8_t* keys_out, uint64_t* off_out, uint8_t* vals_out, cudaStream_t st);

// ---- ppd_dump.cu: the per-txn sub-tries serialised on the GPU ----
// segment kinds IR_SEG_* (seg_b): arena.h
struct IrDumpPlanView {
  // inputs (per block): touched node ids of every IR, and every IR's segments in output order
  const uint32_t* touched;        // concatenated
  const uint32_t* touched_begin;  // [n_ir + 1]
  const uint32_t* seg_a;
  const uint32_t* seg_b;
  const uint32_t* seg_begin;      // [n_ir + 1]
  const uint32_t* seg_end;        // [n_ir], or nullptr: IR i ends where IR i + 1 begins
  const uint32_t* seg_c;          // source offset of IR_SEG_FLAT / IR_SEG_LIT_DEV segments (nullptr: the plan has none)
  const uint8_t* flat;            // the FlatBlock resident in HBM
  const uint8_t* lit;             // the uploaded literal pool
  const uint64_t* ir_base;        // [n_ir] byte offset of the IR in the output (emit only)
  // IRs with more touched slots than a thread block's shared-memory set holds keep their set in HBM: big_off[ir] = word
  // offset of the IR's table in big_scratch (~0: an ordinary IR), big_cap[ir] = its capacity (a power of two); or nullptr
  const uint64_t* big_off;
  const uint32_t* big_cap;
  uint32_t* big_scratch;
  // outputs of ir_size_kernel
  uint32_t* seg_off;              // offset of every segment inside its IR
  uint32_t* ir_size;
  uint32_t* ir_flag;              // 1: the host must serialise this IR
  uint32_t* ir_nuniq;
  uint32_t* u_node;               // [touched_begin[ir] + k]: k-th unique touched node of the IR, its size, its offset
  uint32_t* u_size;
  uint32_t* u_off;
};
void launch_ir_size(const ArenaView& A, const IrDumpPlanView& P, uint32_t n_ir, cudaStream_t st);
// slots of the IR's touched list every key of a txn owns (the device txn loop's walks fill them, txn_core.h)
static const uint32_t MARK_SLOTS = 16;
static const uint32_t IR_SET_MAX_UNIQ = 4096;  // distinct touched nodes an ordinary IR may have (ppd_dump.cu: MAX_UNIQ)
void launch_ir_emit(const ArenaView& A, const IrDumpPlanView& P, uint32_t n_ir, uint8_t* out, cudaStream_t st);

// ---- ppd_parse.cu: compact witness -> instruction list -> tree links -> node arena ----
static const uint32_t PARSE_TILE = 4096;           // bytes per tile of the boundary search
static const uint32_t PARSE_ERR = 0xffffff00u;     // chain values >= PARSE_ERR: PARSE_ERR | PPD_ERR_* of the failing instruction
enum {  // words of ParseBounds::result / ParseTree::result (one 16-word device array)
  PARSE_R_END = 0,     // where the instruction chain from byte 0 ends: n, or PARSE_ERR | code
  PARSE_R_NINS = 1,    // number of instructions
  PARSE_R_FLAG = 2,    // 0, or the first PARSE_WHY_* raised: the host builder must take this witness
  PARSE_R_HEIGHT = 3,  // entries left on the stack (1 for a well-formed witness)
  PARSE_R_ROOT = 4,    // the instruction left on the stack
  PARSE_R_ROOT_ID = 5, // its arena id (written by the emit kernel)
  PARSE_R_NKEYED = 6,  // entries of ParseTree::keyed (leaf, extension and account-leaf instructions)
  PARSE_R_TOTALS = 8,  // PARSE_N_CNT totals of the size counters
  PARSE_R_WORDS = 16
};
enum { PARSE_WHY_DECODE = 1, PARSE_WHY_STACK = 2, PARSE_WHY_NOT_CANONICAL = 3, PARSE_WHY_LEAF_KIND = 4, PARSE_WHY_KEY = 5 };
enum {  // per-instruction size counters, scanned together
  PARSE_C_NODE = 0,   // arena nodes (an account leaf with a non-empty storage trie also owns that trie's NK_ROOT node)
  PARSE_C_HASH = 1,   // hash_pool entries
  PARSE_C_KEY = 2,    // key_pool bytes
  PARSE_C_VAL = 3,    // val_pool bytes (4-byte aligned values)
  PARSE_C_CHILD = 4,  // child_pool slots
  PARSE_C_ACCT = 5,   // account records
  PARSE_C_CODE = 6,   // inline code strings
  PARSE_N_CNT = 7
};
struct ParseBounds {
  const uint8_t* wit;     // witness bytes (readable up to n + 16)
  uint32_t n;
  uint32_t n_tiles, group_tiles, n_groups;
  uint32_t* exit1;        // [n_tiles * PARSE_TILE]
  uint16_t* step1;        // [n_tiles * PARSE_TILE] single-step links inside each tile
  uint32_t* exit2;        // [n_groups * PARSE_TILE]
  uint32_t* group_entry;  // [n_groups]
  uint32_t* tile_entry;   // [n_tiles]
  uint32_t* bitmap;       // [n_tiles * PARSE_TILE / 32]
  uint32_t* tile_count;   // [n_tiles + 1]
  uint32_t* tile_base;    // [n_tiles + 1]
  uint32_t* scan_tmp;     // parse_scan_tmp_words(n_tiles + 1, 1)
  uint32_t* result;       // [PARSE_R_WORDS]
};
struct ParseTree {
  const uint8_t* wit;
  uint32_t n, n_ins;
  const uint32_t* ins_pos;  // [n_ins]
  uint32_t* meta;           // [n_ins]
  uint8_t* knib;            // [n_ins]
  uint32_t* delta;          // [n_ins + 1]
  uint32_t* hb;             // [n_ins + 1]
  int16_t *h16, *m0, *m1, *m2, *m3;  // heights after each instruction; minima over 8 / 64 / 4 096 / 262 144 of them
  uint32_t* parent;         // [n_ins]
  uint32_t* info;           // [n_ins]
  uint32_t* aux0;           // [n_ins]
  uint32_t* keyed;          // [n_ins] the keyed instructions, in no particular order (shape_kernel); result[PARSE_R_NKEYED] of them
  uint32_t *pending, *lvlmax;
  uint32_t *cnt, *scn;      // [PARSE_N_CNT][cnt_stride]
  size_t cnt_stride;        // >= n_ins + 1
  uint32_t* scan_tmp;       // parse_scan_tmp_words(n_ins + 1, PARSE_N_CNT)
  uint32_t* result;
};
struct ParseEmit {
  ParseTree T;
  NodeRec* nodes;
  uint16_t* level;
  uint8_t *key_pool, *val_pool, *hash_pool;
  uint32_t* child_pool;
  AccountRec* accounts;
  uint32_t* acct_list;         // [n_accounts][5]: leaf node, storage trie root id, its NK_ROOT node, flags (1 storage flag, 2 non-empty), code index
  uint64_t* code_se;           // [n_code][2] (begin, end) into the witness
  uint32_t* code_list;         // [n_code][2] (pos, len)
  const uint8_t* code_digest;  // [n_code][32]
  uint32_t n_keyed;            // result[PARSE_R_NKEYED] as the host read it after phase B
};
size_t parse_scan_tmp_words(size_t n, uint32_t K);
uint32_t launch_parse_bounds(const ParseBounds& B, cudaStream_t st);  // the launchers return the number of kernels launched
void launch_parse_scatter(const ParseBounds& B, uint32_t* ins_pos, cudaStream_t st);
uint32_t launch_parse_tree(const ParseTree& T, cudaStream_t st);
void launch_parse_code_list(const ParseEmit& E, cudaStream_t st);
void launch_parse_emit(const ParseEmit& E, cudaStream_t st);

// ---- ppd_txn.cu: the txn loop on the GPU (txn_core.h) ----
void launch_txn_msgs(const txn::View& v, uint64_t* se, cudaStream_t st);
void launch_txn_init(const txn::View& v, const txn::Cursors& init, uint32_t table_slots, cudaStream_t st);
void launch_join(const txn::JoinView& j, cudaStream_t st);
// direct pre-images (j.keep set): the by-address join; slot_owner / slot_best cleared as for launch_join
void launch_join_by_address(const txn::View& v, const txn::JoinView& j, cudaStream_t st);
uint32_t launch_txn_prep(const txn::View& v, const txn::AcctInit& a, uint32_t n_ops1, uint32_t n_ops2, uint32_t max_writes, cudaStream_t st);
// max_keys: the most keys (accessed + written) any txn of the block has; returns the number of launches
// the loops of n blocks as one series of launches (one thread block per task; tasks: device-accessible, e.g. page-locked
// host memory, untouched until the launches have run); max_txns: the most txns any of them has
static const uint32_t LOOP_BATCH_MAX = 12;  // loops per launch (their views travel as kernel parameters)
uint32_t launch_txn_loops(const txn::LoopTask* tasks, uint32_t n, uint32_t max_txns, bool any_shared, cudaStream_t st);
uint32_t txn_loop_uses_shared(uint32_t max_keys);
uint32_t launch_txn_loop(txn::LoopTask* slot, const txn::View& v, uint32_t initial_state, uint32_t max_keys, cudaStream_t st);
void launch_acct_export(const txn::View& v, const txn::JoinView& j, txn::AcctExport* out, cudaStream_t st);

// ---- ppd_microbench.cu ----
bool launch_microbench(int variant, uint32_t* out, uint32_t blocks_per_sm, uint32_t iters, uint32_t* block_threads, double* units_per_thread_iter,
                       cudaStream_t st);

}  // namespace ppd
