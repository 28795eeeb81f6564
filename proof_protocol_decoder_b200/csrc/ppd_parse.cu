// ppd_parse.cu — the compact witness on the GPU: byte stream -> instruction list -> tree links ->
// node arena (north-star items 1 and 2).
//
// Replaces, for a well-formed canonical witness, the reference's
//   WitnessBytes::process_into_instructions_and_header  compact_prestate_processing.rs:683-875
//   ParserState::parse (the rule engine == a stack machine) compact_prestate_processing.rs:325-668
//   create_partial_trie_from_compact_node_rec              compact_to_partial_trie.rs:37-139
//   convert_account_node_data_to_rlp_bytes...              compact_to_partial_trie.rs:141-165
// Anything else (a parse or stack error, a witness whose tree is not the canonical trie of its items,
// a leaf of the wrong kind) is only DETECTED here (`result[R_FLAG]`); the caller then takes the host
// builder, which reproduces the reference's error order exactly.
//
// Phase A: instruction boundaries.  The stream is serial (an instruction's length is known only after
//   its CBOR heads are read), so every byte position is decoded speculatively: nxt[p] = where the
//   instruction that would start at p ends (only a byte below 7 can start one: those positions are listed and
//   decoded, every other position gets the "not an opcode" default).  Per 4 KiB tile (staged in shared memory) the chain
//   p -> nxt[p] is pointer-doubled into exit1[p] = the first position outside the tile that the chain
//   from p reaches; the single-step links are kept too (step1).  Tiles are grouped (about sqrt(#tiles)
//   per group); every position of a group's first tile walks exit1 to the end of the group (exit2); one
//   thread then hops group to group from position 0, the groups' true entries are walked back down to
//   tile entries, and one thread per tile follows step1 from the tile's entry and marks the true
//   instruction starts in a bitmap.  Counts are scanned and the starts scattered into ins_pos[].
// Phase B: the stack machine in closed form.  Every instruction pushes one entry and pops `pops`;
//   height_after = inclusive scan of (1 - pops).  The parent of instruction i is the next instruction
//   whose height_after is not larger (nearest-smaller-value query on a min-pyramid), and i is its
//   (height_after(i) - height_after(parent))-th popped entry: the k-th set bit of a branch mask, or the
//   code / storage slot of an account leaf.  Depths and trie membership come from walking the parent
//   chain (<= 64 steps); seven per-instruction size counters are scanned together; the keyed instructions
//   (leaf, extension, account leaf) are listed.
// Phase C: emit.  Every instruction writes its own arena records (child slot, hashed-out node, branch record in
//   emit_kernel; node, key, value, account record, storage ROOT node of the listed keyed instructions in
//   emit_keyed_kernel); levels are computed by climbing from the leaves with a pending-children counter per
//   inner node (the last child to arrive continues upwards).
#include <cstdint>

#include "../../include/ppd_flat.h"
#include "../../include/ppd_status.h"
#include "arena.h"
#include "ppd_kernels.h"

namespace ppd {

namespace {

constexpr uint32_t TILE = PARSE_TILE;
constexpr uint32_t PERR = PARSE_ERR;
constexpr uint32_t NONE = 0xffffffffu;
constexpr uint32_t HASH_BASE = 0x80000000u;

__constant__ uint8_t C_EMPTY_TRIE_HASH[32] = {0x56, 0xe8, 0x1f, 0x17, 0x1b, 0xcc, 0x55, 0xa6, 0xff, 0x83, 0x45, 0xe6, 0x92, 0xc0, 0xf8, 0x6e,
                                              0x5b, 0x48, 0xe0, 0x1b, 0x99, 0x6c, 0xad, 0xc0, 0x01, 0x62, 0x2f, 0xb5, 0xe3, 0x63, 0xb4, 0x21};
__constant__ uint8_t C_EMPTY_CODE_HASH[32] = {0xc5, 0xd2, 0x46, 0x01, 0x86, 0xf7, 0x23, 0x3c, 0x92, 0x7e, 0x7d, 0xb2, 0xdc, 0xc7, 0x03, 0xc0,
                                              0xe5, 0x00, 0xb6, 0x53, 0xca, 0x82, 0x27, 0x3b, 0x7b, 0xfa, 0xd8, 0x04, 0x5d, 0x85, 0xa4, 0x70};

// ---------------------------------------------------------------------------------------------
// Instruction decode (the byte grammar of compact_prestate_processing.rs:744-875; same checks in the
// same order as the host parser)
// ---------------------------------------------------------------------------------------------
struct Ins {
  uint32_t op, next, flags, aux;
  uint32_t key_pos, key_len, val_pos, val_len;  // val: leaf value / code bytes / balance bytes
  uint64_t nonce;
};

__device__ __forceinline__ bool cbor_head(const uint8_t* w, uint32_t n, uint32_t& pos, uint32_t& major, uint64_t& arg) {
  if (pos >= n) return false;
  uint32_t b = w[pos++];
  major = b >> 5;
  uint32_t ai = b & 31;
  if (ai < 24) {
    arg = ai;
    return true;
  }
  if (ai > 27) return false;
  uint32_t wd = 1u << (ai - 24);
  if (n - pos < wd) return false;
  arg = 0;
  for (uint32_t i = 0; i < wd; i++) arg = (arg << 8) | w[pos++];
  return true;
}
__device__ __forceinline__ bool cbor_bytes(const uint8_t* w, uint32_t n, uint32_t& pos, uint32_t& at, uint32_t& len) {
  uint32_t major;
  uint64_t arg;
  if (!cbor_head(w, n, pos, major, arg) || major != 2 || arg > (uint64_t)(n - pos)) return false;
  at = pos, len = (uint32_t)arg;
  pos += len;
  return true;
}
__device__ __forceinline__ bool key_too_long(uint32_t key_len) { return key_len >= 2 && 2 * (key_len - 1) > 64 + 1; }

// 0, or the PPD_ERR_* code the host parser reports for an instruction starting at p (p < n)
__device__ __forceinline__ uint32_t decode_ins(const uint8_t* w, uint32_t n, uint32_t p, Ins& o) {
  uint32_t pos = p + 1, major;
  uint64_t arg;
  o.op = w[p];
  o.flags = 0, o.aux = 0, o.key_pos = o.key_len = o.val_pos = o.val_len = 0, o.nonce = 0;
  switch (o.op) {
    case PPD_OP_LEAF:
      if (!cbor_bytes(w, n, pos, o.key_pos, o.key_len)) return PPD_ERR_INVALID_BYTE_VECTOR;
      if (key_too_long(o.key_len)) return PPD_ERR_KEY_ERROR;
      if (!cbor_bytes(w, n, pos, o.val_pos, o.val_len)) return PPD_ERR_INVALID_BYTE_VECTOR;
      break;
    case PPD_OP_EXTENSION:
      if (!cbor_bytes(w, n, pos, o.key_pos, o.key_len)) return PPD_ERR_INVALID_BYTE_VECTOR;
      if (key_too_long(o.key_len)) return PPD_ERR_KEY_ERROR;
      break;
    case PPD_OP_BRANCH:
      if (!cbor_head(w, n, pos, major, arg) || major != 0 || arg > 0xffffffffull) return PPD_ERR_INVALID_BYTES_FOR_TYPE;
      o.aux = (uint32_t)arg;
      break;
    case PPD_OP_HASH:
      if (n - pos < 32) return PPD_ERR_INVALID_BYTES_FOR_TYPE;
      o.val_pos = pos, o.val_len = 32;
      pos += 32;
      break;
    case PPD_OP_CODE:
      if (!cbor_bytes(w, n, pos, o.val_pos, o.val_len)) return PPD_ERR_INVALID_BYTES_FOR_TYPE;
      break;
    case PPD_OP_ACCOUNT_LEAF:
      if (!cbor_bytes(w, n, pos, o.key_pos, o.key_len)) return PPD_ERR_INVALID_BYTE_VECTOR;
      if (key_too_long(o.key_len)) return PPD_ERR_KEY_ERROR;
      if (pos >= n) return PPD_ERR_UNEXPECTED_END_OF_STREAM;
      o.flags = w[pos++];
      if (o.flags & 4) {
        if (!cbor_head(w, n, pos, major, arg) || major != 0) return PPD_ERR_INVALID_BYTES_FOR_TYPE;
        o.nonce = arg;
      }
      if (o.flags & 8) {
        if (!cbor_bytes(w, n, pos, o.val_pos, o.val_len) || o.val_len > 32) return PPD_ERR_INVALID_BYTE_VECTOR;
      }
      if (o.flags & 1) {
        if (!cbor_head(w, n, pos, major, arg) || major != 0) return PPD_ERR_INVALID_BYTES_FOR_TYPE;
      }
      break;
    case PPD_OP_EMPTY_ROOT:
      break;
    default:
      return PPD_ERR_INVALID_OPERATOR;
  }
  o.next = pos;
  return 0;
}
// key_bytes_to_nibbles (compact_prestate_processing.rs:1338-1390): number of nibbles of a compact key
__device__ __forceinline__ uint32_t key_nibble_count(const uint8_t* __restrict__ w, uint32_t at, uint32_t len) {
  if (len == 0) return 0;
  if (len == 1) return 1;
  return 2 * (len - 1) - (__ldg(w + at) & 1u);
}
__device__ __forceinline__ void set_nib(uint8_t* pk, uint32_t d, uint32_t nib) { pk[d >> 1] |= (uint8_t)((d & 1) ? nib : (nib << 4)); }
// the key's nibbles written at nibble positions d, d+1, ... of the packed path (caller bounds d + count <= 64)
__device__ __forceinline__ void put_key_nibbles(uint8_t* pk, uint32_t d, const uint8_t* __restrict__ w, uint32_t at, uint32_t len) {
  if (len == 0) return;
  if (len == 1) {
    set_nib(pk, d, __ldg(w + at) & 15u);
    return;
  }
  uint32_t cnt = 2 * (len - 1) - (__ldg(w + at) & 1u);
  for (uint32_t i = 0; i < cnt; i++) {
    uint32_t b = __ldg(w + at + 1 + (i >> 1));
    set_nib(pk, d + i, (i & 1) ? (b & 15u) : (b >> 4));
  }
}
__device__ __forceinline__ uint32_t nth_set_bit(uint32_t mask, uint32_t k) {
  for (uint32_t i = 0; i < k; i++) mask &= mask - 1;
  return mask ? (uint32_t)__ffs(mask) - 1 : 0u;
}

// ---------------------------------------------------------------------------------------------
// Phase A
// ---------------------------------------------------------------------------------------------
constexpr int TE_THREADS = 512;
constexpr uint32_t HALO = 128;  // an instruction's CBOR heads lie within 103 bytes of its opcode

// the tile's bytes (plus halo) staged in shared memory with 128-bit loads; `sb - base` is then indexed by
// absolute stream position exactly like the global witness
__device__ __forceinline__ void stage_tile(uint8_t* sb, const uint8_t* __restrict__ w, uint32_t n, uint32_t base, uint32_t tid, uint32_t nthreads) {
  // base is a multiple of TILE and the witness buffer is 256-byte aligned and readable (zeroed) up to n + 64
  const uint4* src = reinterpret_cast<const uint4*>(w + base);
  uint4* dst = reinterpret_cast<uint4*>(sb);
  const uint32_t avail = ((uint64_t)base + TILE + HALO <= (uint64_t)n + 48) ? (TILE + HALO) / 16 : (n + 48 - base) / 16;
  for (uint32_t k = tid; k < (TILE + HALO) / 16; k += nthreads) dst[k] = k < avail ? __ldg(src + k) : make_uint4(0, 0, 0, 0);
}

// Only a byte below 7 can start an instruction, and 97 % of a witness is hash bytes, so the kernel works on LISTS
// instead of classifying every position (a kernel that classified every position, measured in round 1: 15 k warp
// instructions per tile, most of them single-lane calls of the long decode):
//   pass 1  eight positions per thread: the link tables get their defaults ("not an opcode") with 128-bit stores, the
//           bytes below 7 are found with one exact SIMD-in-register test per word and listed (about 230 per tile);
//   pass 2  one listed position per thread: hashed-out node -> p + 33, empty root -> p + 1, any other opcode must be
//           followed by a CBOR head of the right major type (else the error decode_ins reports); what passes is
//           listed again (about 50 per tile);
//   pass 3  decode_ins, one listed position per thread, so the warps that run the long decode are full;
// then the pointer doubling over the positions whose instruction ends inside the tile.
constexpr uint32_t TE_SMEM_BYTES = 4 * TILE + 4 * 2 * TILE + (TILE + HALO) + 16;

// Four resident thread blocks per SM (32 registers, a few spilled words in the long decode): 0.820-0.825 ms of parse
// device time for one config-2 block alone, against 0.833-0.839 ms with three.
__global__ void __launch_bounds__(TE_THREADS, 4) tile_exit_kernel(const uint8_t* __restrict__ w, uint32_t n, uint32_t* __restrict__ exit1,
                                                                  uint16_t* __restrict__ step1) {
  extern __shared__ __align__(16) uint8_t te_smem[];
  uint32_t* nxt = reinterpret_cast<uint32_t*>(te_smem);            // [TILE]
  uint16_t* step = reinterpret_cast<uint16_t*>(te_smem + 4 * TILE);  // [TILE] single-step links inside the tile (0xffff: the instruction ends outside), for tile_mark_thin_kernel
  uint16_t* active = step + TILE;                                  // [TILE] positions whose chain has not left the tile yet
  uint16_t* cand = active + TILE;                                  // [TILE] positions holding a byte below 7
  uint16_t* slow = cand + TILE;                                    // [TILE] positions that need the long decode
  uint8_t* sb = reinterpret_cast<uint8_t*>(slow + TILE);           // [TILE + HALO]
  uint32_t* counters = reinterpret_cast<uint32_t*>(sb + TILE + HALO);
  uint32_t &n_active = counters[0], &n_cand = counters[1], &n_slow = counters[2];
  constexpr uint32_t SLOW = PERR | 0xfeu;
  constexpr uint32_t NOT_OP = PERR | PPD_ERR_INVALID_OPERATOR;
  const uint32_t base = blockIdx.x * TILE, end = min(base + TILE, n);
  stage_tile(sb, w, n, base, threadIdx.x, TE_THREADS);
  if (threadIdx.x < 3) counters[threadIdx.x] = 0;
  __syncthreads();
  const uint8_t* ws = sb - base;
  // pass 1
  {
    static_assert(TILE == 8 * TE_THREADS, "eight positions per thread");
    const uint32_t o0 = 8 * threadIdx.x;
    const uint2 W = reinterpret_cast<const uint2*>(sb)[threadIdx.x];
    if (base + TILE <= end) {
      const uint4 d = make_uint4(NOT_OP, NOT_OP, NOT_OP, NOT_OP);
      reinterpret_cast<uint4*>(nxt + o0)[0] = d, reinterpret_cast<uint4*>(nxt + o0)[1] = d;
    } else {  // the last tile: positions past the end of the stream are never referenced
#pragma unroll
      for (uint32_t j = 0; j < 8; j++) nxt[o0 + j] = base + o0 + j < end ? NOT_OP : PERR;
    }
    *reinterpret_cast<uint4*>(step + o0) = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    // bit 8k+7 set <=> byte k of the word is below 7: (b | 0x80) - 7 never borrows from the next byte, and its top bit
    // is clear exactly when b < 7 or 128 <= b < 135; the second case has the top bit of b set
    uint32_t m0 = ~(((W.x | 0x80808080u) - 0x07070707u) | W.x) & 0x80808080u;
    uint32_t m1 = ~(((W.y | 0x80808080u) - 0x07070707u) | W.y) & 0x80808080u;
    if (base == 0 && threadIdx.x == 0) m0 |= 0x80u;  // byte 0 is the header: it "ends" at 1 whatever it holds
    while (m0) {
      const uint32_t o = o0 + (((uint32_t)__ffs(m0) - 1u) >> 3);
      m0 &= m0 - 1;
      if (base + o < end) cand[atomicAdd(&n_cand, 1u)] = (uint16_t)o;
    }
    while (m1) {
      const uint32_t o = o0 + 4 + (((uint32_t)__ffs(m1) - 1u) >> 3);
      m1 &= m1 - 1;
      if (base + o < end) cand[atomicAdd(&n_cand, 1u)] = (uint16_t)o;
    }
  }
  __syncthreads();
  // pass 2
  {
    const uint32_t nc = n_cand;
    for (uint32_t a = threadIdx.x; a < nc; a += TE_THREADS) {
      const uint32_t o = cand[a], p = base + o;
      const uint32_t op = ws[p], b1 = ws[p + 1];
      // opcodes 0 1 2 4 5 start with a CBOR head: an unsigned integer (major 0) for a branch mask, else a byte
      // string (major 2); additional info above 27 is not accepted.  Error code per opcode from a nibble table.
      const bool is_uint_head = op == PPD_OP_BRANCH;
      const uint32_t e_head = (((uint32_t)PPD_ERR_INVALID_BYTE_VECTOR * 0x00100011u + (uint32_t)PPD_ERR_INVALID_BYTES_FOR_TYPE * 0x00010100u) >> (4 * (op & 7u))) & 15u;
      const bool head_ok = p + 1 < n && (b1 - (is_uint_head ? 0u : 0x40u)) <= 0x1bu;
      uint32_t r = head_ok ? SLOW : (PERR | e_head);
      r = op == PPD_OP_HASH ? (n - (p + 1) < 32 ? (PERR | PPD_ERR_INVALID_BYTES_FOR_TYPE) : p + 33) : r;
      r = op == PPD_OP_EMPTY_ROOT ? p + 1 : r;
      r = op > PPD_OP_EMPTY_ROOT ? NOT_OP : r;
      r = p == 0 ? 1u : r;
      if (r == SLOW) {
        slow[atomicAdd(&n_slow, 1u)] = (uint16_t)o;
      } else {
        nxt[o] = r;
        if (r < end) {
          step[o] = (uint16_t)(r - base);
          active[atomicAdd(&n_active, 1u)] = (uint16_t)o;
        }
      }
    }
  }
  __syncthreads();
  // pass 3
  {
    const uint32_t ns = n_slow;
    for (uint32_t a = threadIdx.x; a < ns; a += TE_THREADS) {
      const uint32_t o = slow[a];
      Ins ins;
      const uint32_t e = decode_ins(ws, n, base + o, ins);
      const uint32_t r = e ? (PERR | e) : ins.next;
      nxt[o] = r;
      if (r < end) {
        step[o] = (uint16_t)(r - base);
        active[atomicAdd(&n_active, 1u)] = (uint16_t)o;
      }
    }
  }
  __syncthreads();
  // pointer doubling over the few positions that decode to an instruction ending inside the tile; any
  // intermediate value is a point of the same chain, so updating in place is safe
  const uint32_t na = n_active;
  for (;;) {
    bool moved = false;
    for (uint32_t a = threadIdx.x; a < na; a += TE_THREADS) {
      uint32_t o = active[a], x = nxt[o];
      if (x < end) {
        nxt[o] = nxt[x - base];
        moved = true;
      }
    }
    if (!__syncthreads_or(moved)) break;
  }
  {
    const uint4* s4 = reinterpret_cast<const uint4*>(nxt);
    uint4* d4 = reinterpret_cast<uint4*>(exit1 + base);  // the exit1 array is padded to whole tiles
#pragma unroll
    for (uint32_t k = threadIdx.x; k < TILE / 4; k += TE_THREADS) d4[k] = s4[k];
  }
  // the whole 8 KiB link table of the tile (entries past the end of the stream are never followed)
  reinterpret_cast<uint4*>(step1 + (size_t)base)[threadIdx.x] = reinterpret_cast<const uint4*>(step)[threadIdx.x];
}

// exit2[g][c]: where the chain from position c of group g's first tile leaves the group
__global__ void group_exit_kernel(const uint32_t* __restrict__ exit1, uint32_t n, uint32_t group_bytes, uint32_t* __restrict__ exit2) {
  uint32_t g = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t gb = (uint64_t)g * group_bytes;
  uint32_t gend = (uint32_t)min((uint64_t)n, gb + group_bytes);
  uint32_t p = (uint32_t)gb + c;
  if (c >= TILE || p >= gend) return;
  uint32_t v = p;
  while (v < gend) v = __ldg(exit1 + v);
  exit2[(size_t)g * TILE + c] = v;
}

// hop group to group from position 0; result[0] = n (clean end) or PERR | code
__global__ void top_chain_kernel(const uint32_t* __restrict__ exit1, const uint32_t* __restrict__ exit2, uint32_t n, uint32_t group_bytes,
                                 uint32_t* __restrict__ group_entry, uint32_t* __restrict__ result) {
  if (blockIdx.x || threadIdx.x) return;
  uint32_t cur = 0;
  while (cur < n) {
    uint32_t g = cur / group_bytes;
    uint64_t gb = (uint64_t)g * group_bytes;
    uint32_t gend = (uint32_t)min((uint64_t)n, gb + group_bytes);
    group_entry[g] = cur;
    uint32_t off = cur - (uint32_t)gb;
    if (off < TILE) {
      cur = exit2[(size_t)g * TILE + off];
    } else {  // an instruction jumped over the group's first tile
      while (cur < gend) cur = exit1[cur];
    }
  }
  result[PARSE_R_END] = cur;
}

__global__ void tile_entry_kernel(const uint32_t* __restrict__ exit1, const uint32_t* __restrict__ group_entry, uint32_t n, uint32_t n_groups,
                                  uint32_t group_bytes, uint32_t* __restrict__ tile_entry) {
  uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  uint32_t cur = group_entry[g];
  if (cur == NONE) return;
  uint32_t gend = (uint32_t)min((uint64_t)n, (uint64_t)g * group_bytes + group_bytes);
  while (cur < gend) {
    tile_entry[cur / TILE] = cur;
    cur = __ldg(exit1 + cur);
  }
}

// One thread per tile follows the tile's single-step links (written by tile_exit_kernel) from the tile's true entry,
// straight from the global link table, and marks the instruction starts (the bitmap is zeroed beforehand and only
// the words that hold a start are written).  A walk is about 124 dependent 2-byte loads, so a lone launch takes longer
// than one warp per tile with the links staged in shared memory (88 vs 36 us), but it issues 40x fewer warp
// instructions (no 8 KiB staging per tile, 32 walks per warp instead of one), and with other blocks' kernels beside it
// the parse is bound by issue slots, not by latency.
__global__ void __launch_bounds__(128) tile_mark_thin_kernel(const uint16_t* __restrict__ step1, uint32_t n_tiles, const uint32_t* __restrict__ tile_entry,
                                                             uint32_t* __restrict__ bitmap, uint32_t* __restrict__ tile_count) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  const uint32_t cur = tile_entry[t];
  uint32_t count = 0;
  if (cur != NONE) {
    const uint16_t* __restrict__ step = step1 + (size_t)t * TILE;
    uint32_t* __restrict__ bits = bitmap + (size_t)t * (TILE / 32);
    uint32_t o = cur - t * TILE;
    if (cur == 0) o = __ldg(step);  // the header byte is not an instruction
    uint32_t word = o >> 5, acc = 0;  // starts are visited in increasing order
    while (o != 0xffffu) {
      if ((o >> 5) != word) {
        bits[word] = acc;
        word = o >> 5, acc = 0;
      }
      acc |= 1u << (o & 31);
      count++;
      o = __ldg(step + o);
    }
    if (acc) bits[word] = acc;
  }
  tile_count[t] = count;
}

__global__ void __launch_bounds__(TILE / 32) ins_scatter_kernel(const uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ tile_base,
                                                                uint32_t* __restrict__ ins_pos) {
  __shared__ uint32_t wsum[TILE / 32 / 32];
  const uint32_t t = blockIdx.x, tid = threadIdx.x;
  uint32_t word = bitmap[(size_t)t * (TILE / 32) + tid];
  uint32_t c = __popc(word), incl = c;
  for (int off = 1; off < 32; off <<= 1) {
    uint32_t x = __shfl_up_sync(0xffffffffu, incl, off);
    if ((tid & 31) >= (uint32_t)off) incl += x;
  }
  if ((tid & 31) == 31) wsum[tid >> 5] = incl;
  __syncthreads();
  uint32_t before = 0;
  for (uint32_t k = 0; k < (tid >> 5); k++) before += wsum[k];
  uint32_t at = tile_base[t] + before + incl - c;
  const uint32_t p0 = t * TILE + tid * 32;
  while (word) {
    uint32_t b = (uint32_t)__ffs(word) - 1;
    word &= word - 1;
    ins_pos[at++] = p0 + b;
  }
}

// ---------------------------------------------------------------------------------------------
// multi-array exclusive scan: K arrays of n uint32 each, array k at in + k * stride
// ---------------------------------------------------------------------------------------------
constexpr int MS_B = 256, MS_ITEMS = 4, MS_ELEMS = MS_B * MS_ITEMS;

__global__ void __launch_bounds__(MS_B) mscan_block_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t n, size_t stride,
                                                           uint32_t* __restrict__ block_sums, size_t sums_stride) {
  __shared__ uint32_t warp_sums[MS_B / 32];
  const uint32_t k = blockIdx.y;
  in += k * stride, out += k * stride;
  uint32_t base = blockIdx.x * MS_ELEMS + threadIdx.x * MS_ITEMS;
  uint32_t v[MS_ITEMS], sum = 0;
#pragma unroll
  for (int q = 0; q < MS_ITEMS; q++) {
    v[q] = base + q < n ? in[base + q] : 0u;
    sum += v[q];
  }
  uint32_t incl = sum;
  for (int off = 1; off < 32; off <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, incl, off);
    if ((threadIdx.x & 31) >= (uint32_t)off) incl += t;
  }
  if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = incl;
  __syncthreads();
  if (threadIdx.x < 32) {
    uint32_t ws = threadIdx.x < MS_B / 32 ? warp_sums[threadIdx.x] : 0u, wi = ws;
    for (int off = 1; off < 32; off <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, wi, off);
      if (threadIdx.x >= (uint32_t)off) wi += t;
    }
    if (threadIdx.x < MS_B / 32) warp_sums[threadIdx.x] = wi - ws;
    if (threadIdx.x == MS_B / 32 - 1 && block_sums) block_sums[k * sums_stride + blockIdx.x] = wi;
  }
  __syncthreads();
  uint32_t excl = incl - sum + warp_sums[threadIdx.x >> 5];
#pragma unroll
  for (int q = 0; q < MS_ITEMS; q++) {
    if (base + q < n) out[base + q] = excl;
    excl += v[q];
  }
}
__global__ void __launch_bounds__(MS_B) mscan_add_kernel(uint32_t* __restrict__ out, uint32_t n, size_t stride, const uint32_t* __restrict__ block_offsets,
                                                         size_t sums_stride) {
  const uint32_t k = blockIdx.y;
  out += k * stride;
  uint32_t add = block_offsets[k * sums_stride + blockIdx.x];
  uint32_t i = blockIdx.x * MS_ELEMS + threadIdx.x;
#pragma unroll
  for (int q = 0; q < MS_ITEMS; q++) {
    uint32_t j = i + q * MS_B;
    if (j < n) out[j] += add;
  }
}

// returns the number of kernels launched
uint32_t mscan(const uint32_t* in, uint32_t* out, uint32_t n, size_t stride, uint32_t K, uint32_t* tmp, cudaStream_t st) {
  if (!n) return 0;
  uint32_t nb = (n + MS_ELEMS - 1) / MS_ELEMS, launches = 1;
  size_t ss = (nb + 3) & ~(size_t)3;
  mscan_block_kernel<<<dim3(nb, K), MS_B, 0, st>>>(in, out, n, stride, nb > 1 ? tmp : nullptr, ss);
  if (nb > 1) {
    launches += mscan(tmp, tmp, nb, ss, K, tmp + K * ss, st);
    mscan_add_kernel<<<dim3(nb, K), MS_B, 0, st>>>(out, n, stride, tmp, ss);
    launches++;
  }
  return launches;
}

// ---------------------------------------------------------------------------------------------
// Phase B
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t dw0(uint32_t kind, uint32_t nib_start, uint32_t nib_len) { return kind | (nib_start << 8) | (nib_len << 16); }
__device__ __forceinline__ void raise(uint32_t* result, uint32_t reason) { atomicCAS(result + PARSE_R_FLAG, 0u, reason); }

__device__ __forceinline__ uint32_t pops_of(uint32_t meta) {
  uint32_t op = meta & 7u;
  if (op == PPD_OP_EXTENSION) return 1;
  if (op == PPD_OP_BRANCH) return __popc(meta >> 16);
  if (op == PPD_OP_ACCOUNT_LEAF) return ((meta >> 8) & 1u) + ((meta >> 9) & 1u);
  return 0;
}

// meta = op | flags << 8 | (branch mask & 0xffff) << 16
__device__ __forceinline__ void ins_info_one(const ParseTree& T, uint32_t i) {
  if (i == T.n_ins) {
    T.delta[i] = 0;
    return;
  }
  Ins o;
  uint32_t e = decode_ins(T.wit, T.n, T.ins_pos[i], o);
  if (e || o.op > 6) {
    raise(T.result, PARSE_WHY_DECODE);
    o.op = PPD_OP_EMPTY_ROOT, o.flags = 0, o.aux = 0, o.key_len = 0;
  }
  if (o.op == PPD_OP_BRANCH && (o.aux >> 16)) raise(T.result, PARSE_WHY_STACK);
  uint32_t meta = o.op | ((o.flags & 0xffu) << 8) | ((o.aux & 0xffffu) << 16);
  T.meta[i] = meta;
  uint32_t kn = key_nibble_count(T.wit, o.key_pos, o.key_len);
  T.knib[i] = (uint8_t)min(kn, 255u);
  uint32_t pops = pops_of(meta);
  T.delta[i] = 1u - pops;
  T.pending[i] = o.op == PPD_OP_ACCOUNT_LEAF ? ((o.flags >> 1) & 1u) : pops;
  T.lvlmax[i] = 0;
  T.aux0[i] = NONE;
}
__global__ void ins_info_kernel(ParseTree T) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > T.n_ins) return;
  ins_info_one(T, i);
}

// heights as int16 (+ sentinel), stack underflow check
__global__ void heights_kernel(ParseTree T) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > T.n_ins) return;
  if (i == T.n_ins) {
    T.h16[i] = INT16_MIN;
    T.result[PARSE_R_HEIGHT] = T.hb[i];
    return;
  }
  int32_t hb = (int32_t)T.hb[i];
  int32_t pops = (int32_t)pops_of(T.meta[i]);
  if (hb < pops) raise(T.result, PARSE_WHY_STACK);
  int32_t ha = hb + 1 - pops;
  if (ha > 30000 || ha < 1) {
    raise(T.result, PARSE_WHY_STACK);
    ha = ha < 1 ? 1 : 30000;
  }
  T.h16[i] = (int16_t)ha;
}

__global__ void min64_i16_kernel(const int16_t* __restrict__ in, uint32_t n_in, int16_t* __restrict__ out, uint32_t n_out) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_out) return;
  int m = INT16_MAX;
  uint32_t lo = j * 64, hi = min(lo + 64, n_in);
  for (uint32_t k = lo; k < hi; k++) m = min(m, (int)in[k]);
  out[j] = (int16_t)m;
}

// m0[c] = min of in[8c .. 8c + 7], m1[j] = min of in[64j .. 64j + 63]: one thread per cell of 64, eight 128-bit loads
// (the arrays are carved at 256-byte boundaries inside one allocation, so a whole cell is always readable)
__global__ void min8_64_i16_kernel(const int16_t* __restrict__ in, uint32_t n_in, int16_t* __restrict__ m0, int16_t* __restrict__ m1, uint32_t n_m1) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_m1) return;
  int m = INT16_MAX;
  uint32_t packed[4];
#pragma unroll
  for (uint32_t c = 0; c < 8; c++) {
    const uint32_t lo = j * 64 + c * 8;
    int mc = INT16_MAX;
    if (lo < n_in) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(in + lo));
      const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (uint32_t q = 0; q < 4; q++) {
        const int a = (int)(int16_t)(wv[q] & 0xffffu), b = (int)(int16_t)(wv[q] >> 16);
        if (lo + 2 * q < n_in) mc = min(mc, a);
        if (lo + 2 * q + 1 < n_in) mc = min(mc, b);
      }
    }
    m = min(m, mc);
    const uint32_t h = (uint32_t)mc & 0xffffu;
    packed[c >> 1] = (c & 1) ? (packed[c >> 1] | (h << 16)) : h;
  }
  reinterpret_cast<uint4*>(m0)[j] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
  m1[j] = (int16_t)m;
}

// smallest r > q with h16[r] < thr, over the pyramid with an extra 8-wide level (h16[n_ins] = INT16_MIN ends every
// scan).  A scan that has to jump a sibling subtree of a few hundred instructions takes at most 7 single steps and
// 7 steps of eight on either side of its steps of 64, instead of up to 63 single steps on either side.
__device__ __forceinline__ uint32_t scan_right8(const ParseTree& T, uint32_t q, int thr) {
  uint32_t p = q + 1;
  for (;;) {
    if ((p & 7u) == 0u) {
      if ((p & 63u) == 0u) {
        if ((p & 4095u) == 0u) {
          if ((p & 262143u) == 0u && T.m3[p >> 18] >= thr) {
            p += 262144u;
            continue;
          }
          if (T.m2[p >> 12] >= thr) {
            p += 4096u;
            continue;
          }
        }
        if (T.m1[p >> 6] >= thr) {
          p += 64u;
          continue;
        }
      }
      if (T.m0[p >> 3] >= thr) {
        p += 8u;
        continue;
      }
    }
    if (T.h16[p] < thr) return p;
    p++;
  }
}

// info = slot (bits 0-3) | role (bits 4-5: 0 child of branch / extension, 1 account code, 2 account storage)
//        | depth << 8 | in_storage << 16 | storage_nonempty << 17 (account leaves)
__global__ void link_kernel16(ParseTree T) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T.n_ins) return;
  int ha = T.h16[i];
  const uint32_t j = scan_right8(T, i, ha + 1);  // first j > i with height_after(j) <= height_after(i); n_ins when none
  T.parent[i] = j;
  uint32_t info = 0;
  if (j < T.n_ins) {
    uint32_t pm = T.meta[j], pop = pm & 7u, cop = T.meta[i] & 7u;
    uint32_t k = (uint32_t)(ha - (int)T.h16[j]);
    if (k >= pops_of(pm)) {
      raise(T.result, PARSE_WHY_STACK);
      k = 0;
    }
    uint32_t role = 0;
    if (pop == PPD_OP_ACCOUNT_LEAF) {
      bool has_code = (pm >> 8) & 1u;
      role = (has_code && k == 0) ? 1u : 2u;
      if (role == 1) {
        if (cop != PPD_OP_CODE && cop != PPD_OP_HASH) raise(T.result, PARSE_WHY_STACK);
        T.aux0[j] = i;
      } else if (cop == PPD_OP_CODE) {
        raise(T.result, PARSE_WHY_STACK);
      }
    } else if (cop == PPD_OP_CODE || cop == PPD_OP_EMPTY_ROOT) {
      raise(T.result, PARSE_WHY_NOT_CANONICAL);  // an empty child of a branch / extension: the host rebuilds from the items
    }
    info = k | (role << 4);
  } else {
    uint32_t cop = T.meta[i] & 7u;
    if (cop == PPD_OP_CODE || cop == PPD_OP_EMPTY_ROOT) raise(T.result, PARSE_WHY_NOT_CANONICAL);
    T.result[PARSE_R_ROOT] = i;
  }
  T.info[i] = info;
}

// depth inside the own trie, trie membership, canonicity, per-instruction sizes
__device__ __forceinline__ void shape_one(const ParseTree& T, uint32_t i) {
  const size_t S = T.cnt_stride;
  if (i == T.n_ins) {
    for (int k = 0; k < PARSE_N_CNT; k++) T.cnt[k * S + i] = 0;
    return;
  }
  const uint32_t meta = T.meta[i], op = meta & 7u;
  uint32_t info = T.info[i];
  uint32_t c_node = 0, c_hash = 0, c_key = 0, c_val = 0, c_child = 0, c_acct = 0, c_code = 0;
  if (op == PPD_OP_HASH) {
    c_hash = 1;
  } else if (op == PPD_OP_CODE) {
    c_code = 1;
  } else if (op != PPD_OP_EMPTY_ROOT) {
    // walk to the root of the own trie
    uint32_t cur = i, d = 0, in_storage = 0;
    for (uint32_t guard = 0; guard < 4096; guard++) {
      uint32_t j = T.parent[cur];
      if (j >= T.n_ins) break;
      uint32_t pop = T.meta[j] & 7u;
      if (pop == PPD_OP_BRANCH) {
        d += 1;
      } else if (pop == PPD_OP_EXTENSION) {
        d += T.knib[j];
      } else {
        in_storage = ((T.info[cur] >> 4) & 3u) == 2u;
        break;
      }
      if (d > 200) break;
      cur = j;
    }
    const uint32_t kn = T.knib[i];
    c_node = 1;
    if (op == PPD_OP_BRANCH) {
      if (d >= 64) raise(T.result, PARSE_WHY_KEY);
      uint32_t k = __popc(meta >> 16);
      if (k < 2) raise(T.result, PARSE_WHY_NOT_CANONICAL);
      c_child = k;
    } else {
      if (d + kn > 64) raise(T.result, PARSE_WHY_KEY);
      uint32_t nd = min(d + kn, 64u);
      c_key = (nd + 1) / 2 + 1;
      if (op == PPD_OP_EXTENSION) {
        uint32_t cop = i ? (T.meta[i - 1] & 7u) : 7u;  // the child is the entry on top of the stack: the previous instruction
        if (kn == 0 || !(cop == PPD_OP_BRANCH || cop == PPD_OP_HASH)) raise(T.result, PARSE_WHY_NOT_CANONICAL);
      } else if (op == PPD_OP_LEAF) {
        if (!in_storage) raise(T.result, PARSE_WHY_LEAF_KIND);
        Ins o;
        decode_ins(T.wit, T.n, T.ins_pos[i], o);
        uint32_t vl = o.val_len, hl = 0;
        if (!(vl == 1 && __ldg(T.wit + o.val_pos) < 0x80)) hl = vl < 56 ? 1 : vl < 256 ? 2 : vl < 65536 ? 3 : vl < (1u << 24) ? 4 : 5;
        c_val = (hl + vl + 3) & ~3u;
      } else {  // account leaf
        if (in_storage) raise(T.result, PARSE_WHY_LEAF_KIND);
        c_acct = 1;
        uint32_t nonempty = 0;
        if (meta & (2u << 8)) {
          uint32_t sop = i ? (T.meta[i - 1] & 7u) : 7u;
          if (sop == PPD_OP_HASH) {
            const uint8_t* h = T.wit + T.ins_pos[i - 1] + 1;
            for (int k = 0; k < 32; k++) nonempty |= (uint32_t)(__ldg(h + k) != C_EMPTY_TRIE_HASH[k]);
          } else {
            nonempty = sop != PPD_OP_EMPTY_ROOT;
          }
        }
        c_node += nonempty;  // the NK_ROOT node of the storage trie
        info |= nonempty << 17;
      }
    }
    info |= (min(d, 255u) << 8) | (in_storage << 16);
    T.info[i] = info;
  }
  T.cnt[PARSE_C_NODE * S + i] = c_node;
  T.cnt[PARSE_C_HASH * S + i] = c_hash;
  T.cnt[PARSE_C_KEY * S + i] = c_key;
  T.cnt[PARSE_C_VAL * S + i] = c_val;
  T.cnt[PARSE_C_CHILD * S + i] = c_child;
  T.cnt[PARSE_C_ACCT * S + i] = c_acct;
  T.cnt[PARSE_C_CODE * S + i] = c_code;
}
// One thread per instruction; the keyed instructions (leaf, extension, account leaf: the ones whose path the emit
// phase assembles by a walk up their ancestors) are appended to T.keyed, one global atomic per thread block, so that
// emit_keyed_kernel runs with full warps.  The list's order is the order thread blocks finish in; nothing depends on it.
__global__ void __launch_bounds__(256) shape_kernel(ParseTree T) {
  __shared__ uint32_t n_here, base;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (threadIdx.x == 0) n_here = 0;
  __syncthreads();
  bool keyed = false;
  if (i <= T.n_ins) {
    shape_one(T, i);
    if (i < T.n_ins) {
      const uint32_t op = T.meta[i] & 7u;
      keyed = op == PPD_OP_LEAF || op == PPD_OP_EXTENSION || op == PPD_OP_ACCOUNT_LEAF;
    }
  }
  const uint32_t at = keyed ? atomicAdd(&n_here, 1u) : 0u;
  __syncthreads();
  if (threadIdx.x == 0 && n_here) base = atomicAdd(T.result + PARSE_R_NKEYED, n_here);
  __syncthreads();
  if (keyed) T.keyed[base + at] = i;
}

__global__ void totals_kernel(ParseTree T) {
  uint32_t k = threadIdx.x;
  if (k < PARSE_N_CNT) T.result[PARSE_R_TOTALS + k] = T.scn[k * T.cnt_stride + T.n_ins];
}

// ---------------------------------------------------------------------------------------------
// Phase C
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t id_of(const ParseTree& T, uint32_t i) {
  uint32_t op = T.meta[i] & 7u;
  if (op == PPD_OP_HASH) return HASH_BASE + T.scn[PARSE_C_HASH * T.cnt_stride + i];
  if (op == PPD_OP_CODE || op == PPD_OP_EMPTY_ROOT) return NODE_EMPTY;
  return T.scn[PARSE_C_NODE * T.cnt_stride + i];
}

// inline code: (begin, end) pairs for the keccak launch and (pos, len) for the host
__global__ void code_list_kernel(ParseEmit E) {
  const ParseTree& T = E.T;
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T.n_ins || (T.meta[i] & 7u) != PPD_OP_CODE) return;
  Ins o;
  decode_ins(T.wit, T.n, T.ins_pos[i], o);
  uint32_t c = T.scn[PARSE_C_CODE * T.cnt_stride + i];
  E.code_se[2 * c] = o.val_pos, E.code_se[2 * c + 1] = (uint64_t)o.val_pos + o.val_len;
  E.code_list[2 * c] = o.val_pos, E.code_list[2 * c + 1] = o.val_len;
}

__device__ __forceinline__ void copy_bytes(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n) {
  for (uint32_t k = 0; k < n; k++) dst[k] = __ldg(src + k);
}

// One instruction in twenty carries a key (leaf, extension, account leaf) and needs its path assembled by a walk up
// its ancestors; with one instruction per thread those few lanes set every warp's instruction count (round-1 capture:
// 6 of 32 threads active, 58 M warp instructions).  emit_kernel does the short work of every instruction (child slot
// of the parent branch, hashed-out node, branch record); emit_keyed_kernel takes the keyed instructions from the
// list shape_kernel made, one per thread.
__device__ __forceinline__ void emit_keyed(const ParseEmit& E, uint32_t i) {
  const ParseTree& T = E.T;
  const size_t S = T.cnt_stride;
  const uint32_t meta = T.meta[i], op = meta & 7u, info = T.info[i];
  const uint32_t pos = T.ins_pos[i];
  const uint32_t my_id = T.scn[PARSE_C_NODE * S + i];
  Ins o;
  decode_ins(T.wit, T.n, pos, o);
  const uint32_t d = (info >> 8) & 255u, kn = T.knib[i], nd = min(d + kn, 64u);
  // the full path: own key nibbles, then every ancestor's contribution up to the root of the own trie
  uint8_t pk[36];
#pragma unroll
  for (int k = 0; k < 36; k++) pk[k] = 0;
  if (d + kn <= 64) put_key_nibbles(pk, d, T.wit, o.key_pos, o.key_len);
  {
    uint32_t cur = i;
    for (uint32_t guard = 0; guard < 4096; guard++) {
      uint32_t j = T.parent[cur];
      if (j >= T.n_ins) break;
      uint32_t pm = T.meta[j], pop = pm & 7u;
      uint32_t pd = (T.info[j] >> 8) & 255u;
      if (pop == PPD_OP_BRANCH) {
        if (pd < 64) set_nib(pk, pd, nth_set_bit(pm >> 16, T.info[cur] & 15u));
      } else if (pop == PPD_OP_EXTENSION) {
        Ins e;
        decode_ins(T.wit, T.n, T.ins_pos[j], e);
        if (pd + T.knib[j] <= 64) put_key_nibbles(pk, pd, T.wit, e.key_pos, e.key_len);
      } else {
        break;
      }
      cur = j;
    }
  }
  const uint32_t koff = T.scn[PARSE_C_KEY * S + i];
  {
    uint8_t* kd = E.key_pool + koff;
    uint32_t nb = (nd + 1) / 2;
    for (uint32_t k = 0; k < nb; k++) kd[k] = pk[k];
    kd[nb] = 0;
  }
  if (op == PPD_OP_EXTENSION) {
    E.nodes[my_id] = NodeRec{dw0(NK_EXT, d, kn), koff, i ? id_of(T, i - 1) : NODE_EMPTY, 0};
    return;
  }
  if (op == PPD_OP_LEAF) {
    // rlp_str(value), compact_to_partial_trie.rs:119
    uint32_t voff = T.scn[PARSE_C_VAL * S + i], vl = o.val_len, hl = 0;
    uint8_t* v = E.val_pool + voff;
    if (!(vl == 1 && __ldg(T.wit + o.val_pos) < 0x80)) {
      if (vl < 56) {
        v[hl++] = (uint8_t)(0x80 + vl);
      } else {
        uint32_t k = vl < 256 ? 1 : vl < 65536 ? 2 : vl < (1u << 24) ? 3 : 4;
        v[hl++] = (uint8_t)(0xb7 + k);
        for (uint32_t q = k; q-- > 0;) v[hl++] = (uint8_t)(vl >> (8 * q));
      }
    }
    copy_bytes(v + hl, T.wit + o.val_pos, vl);
    E.nodes[my_id] = NodeRec{dw0(NK_LEAF, d, kn), koff, voff, hl + vl};
    return;
  }
  // account leaf: the record (compact_to_partial_trie.rs:141-165), the storage trie's ROOT node, the host's list entry
  const uint32_t a = T.scn[PARSE_C_ACCT * S + i];
  const uint32_t nonempty = (info >> 17) & 1u;
  uint32_t sroot = NODE_EMPTY, root_node = NODE_EMPTY;
  if (meta & (2u << 8)) sroot = i ? id_of(T, i - 1) : NODE_EMPTY;
  if (nonempty) {
    root_node = my_id + 1;
    E.nodes[root_node] = NodeRec{dw0(NK_ROOT, 0, 0), 0, sroot, 0};
  }
  {
    uint32_t* r = reinterpret_cast<uint32_t*>(E.accounts + a);
    uint8_t* rb = reinterpret_cast<uint8_t*>(r);
    for (int k = 0; k < 36; k++) r[k] = 0;
    for (int k = 0; k < 8; k++) rb[31 - k] = (uint8_t)(o.nonce >> (8 * k));
    if (meta & (8u << 8)) copy_bytes(rb + 32 + 32 - o.val_len, T.wit + o.val_pos, o.val_len);
    for (int k = 0; k < 32; k++) rb[64 + k] = C_EMPTY_TRIE_HASH[k];
    uint32_t code_idx = NONE;
    if (meta & (1u << 8)) {
      uint32_t ci = T.aux0[i];
      if (ci < T.n_ins) {
        if ((T.meta[ci] & 7u) == PPD_OP_CODE) {
          code_idx = T.scn[PARSE_C_CODE * S + ci];
          const uint8_t* dg = E.code_digest + 32ull * code_idx;
          for (int k = 0; k < 32; k++) rb[96 + k] = dg[k];
        } else {
          copy_bytes(rb + 96, T.wit + T.ins_pos[ci] + 1, 32);
        }
      }
    } else {
      for (int k = 0; k < 32; k++) rb[96 + k] = C_EMPTY_CODE_HASH[k];
    }
    r[32] = root_node;  // storage_src
    uint32_t* L = E.acct_list + 5ull * a;
    L[0] = my_id, L[1] = sroot, L[2] = root_node, L[3] = ((meta >> 9) & 1u) | (nonempty << 1), L[4] = code_idx;
  }
  E.nodes[my_id] = NodeRec{dw0(NK_LEAF_ACCOUNT, d, kn), koff, a, 0};
}

__global__ void __launch_bounds__(256) emit_kernel(ParseEmit E) {
  const ParseTree& T = E.T;
  const size_t S = T.cnt_stride;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T.n_ins) return;
  const uint32_t meta = T.meta[i], op = meta & 7u, info = T.info[i];
  const uint32_t my_id = id_of(T, i);
  // register with the parent branch
  {
    uint32_t j = T.parent[i];
    if (j >= T.n_ins) T.result[PARSE_R_ROOT_ID] = my_id;
    if (j < T.n_ins && (T.meta[j] & 7u) == PPD_OP_BRANCH) E.child_pool[T.scn[PARSE_C_CHILD * S + j] + (info & 15u)] = my_id;
  }
  if (op == PPD_OP_HASH) {
    uint32_t* dst = reinterpret_cast<uint32_t*>(E.hash_pool + 32ull * (my_id - HASH_BASE));
    // 32 bytes at an arbitrary alignment: nine aligned words re-aligned with funnel shifts (the witness
    // buffer is readable past its end)
    const uintptr_t a = reinterpret_cast<uintptr_t>(T.wit + T.ins_pos[i] + 1);
    const uint32_t* q = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(a & 3) * 8;
    uint32_t x[9];
#pragma unroll
    for (int c = 0; c < 9; c++) x[c] = __ldg(q + c);
    uint4 lo = make_uint4(__funnelshift_r(x[0], x[1], sh), __funnelshift_r(x[1], x[2], sh), __funnelshift_r(x[2], x[3], sh), __funnelshift_r(x[3], x[4], sh));
    uint4 hi = make_uint4(__funnelshift_r(x[4], x[5], sh), __funnelshift_r(x[5], x[6], sh), __funnelshift_r(x[6], x[7], sh), __funnelshift_r(x[7], x[8], sh));
    reinterpret_cast<uint4*>(dst)[0] = lo, reinterpret_cast<uint4*>(dst)[1] = hi;
  } else if (op == PPD_OP_BRANCH) {
    E.nodes[my_id] = NodeRec{dw0(NK_BRANCH, 0, 0), T.scn[PARSE_C_CHILD * S + i], meta >> 16, 0};
  }
}
__global__ void __launch_bounds__(128) emit_keyed_kernel(ParseEmit E) {
  const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= E.n_keyed) return;
  emit_keyed(E, E.T.keyed[a]);
}

// levels: 1 + the maximum level of what a node reads (host_arena.h constructors), bottom-up
__global__ void climb_kernel(ParseEmit E) {
  const ParseTree& T = E.T;
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T.n_ins) return;
  const size_t S = T.cnt_stride;
  const uint32_t meta = T.meta[i], op = meta & 7u;
  const bool starter = op == PPD_OP_LEAF || op == PPD_OP_HASH || op == PPD_OP_EMPTY_ROOT || op == PPD_OP_CODE ||
                       (op == PPD_OP_ACCOUNT_LEAF && !(meta & (2u << 8)));
  if (!starter) return;
  if (op == PPD_OP_LEAF || op == PPD_OP_ACCOUNT_LEAF) E.level[T.scn[PARSE_C_NODE * S + i]] = 0;
  uint32_t cur = i, lv = 0;
  for (uint32_t guard = 0; guard < 4096; guard++) {
    uint32_t j = T.parent[cur];
    if (j >= T.n_ins) break;
    uint32_t pm = T.meta[j], pop = pm & 7u;
    uint32_t nid = T.scn[PARSE_C_NODE * S + j];
    if (pop == PPD_OP_ACCOUNT_LEAF) {
      if (((T.info[cur] >> 4) & 3u) != 2u) break;  // the code child does not affect the level
      uint32_t nonempty = (T.info[j] >> 17) & 1u;
      if (nonempty) E.level[nid + 1] = (uint16_t)min(lv + 1, 65535u);
      lv = nonempty ? lv + 2 : 0;
    } else if (pop == PPD_OP_BRANCH || pop == PPD_OP_EXTENSION) {
      if (lv) {  // (lvlmax starts at 0: a level-0 child -- two instructions in three are hashed-out nodes -- has nothing to add)
        atomicMax(T.lvlmax + j, lv);
        __threadfence();
      }
      uint32_t old = atomicSub(T.pending + j, 1u);
      if (old != 1u) break;
      __threadfence();
      lv = atomicMax(T.lvlmax + j, 0u) + 1;
    } else {
      break;
    }
    E.level[nid] = (uint16_t)min(lv, 65535u);
    cur = j;
  }
}

inline uint32_t cdiv(uint64_t a, uint32_t b) { return (uint32_t)((a + b - 1) / b); }

}  // namespace

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
size_t parse_scan_tmp_words(size_t n, uint32_t K) {
  size_t total = 0;
  while (n > 1) {
    n = (n + MS_ELEMS - 1) / MS_ELEMS;
    total += K * ((n + 3) & ~(size_t)3);
  }
  return total + 16;
}

uint32_t launch_parse_bounds(const ParseBounds& B, cudaStream_t st) {
  const uint32_t group_bytes = B.group_tiles * TILE;
  static const bool once = cudaFuncSetAttribute(tile_exit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TE_SMEM_BYTES) == cudaSuccess;
  (void)once;
  tile_exit_kernel<<<B.n_tiles, TE_THREADS, TE_SMEM_BYTES, st>>>(B.wit, B.n, B.exit1, B.step1);
  group_exit_kernel<<<dim3(TILE / 256, B.n_groups), 256, 0, st>>>(B.exit1, B.n, group_bytes, B.exit2);
  cudaMemsetAsync(B.group_entry, 0xff, 4ull * B.n_groups, st);
  cudaMemsetAsync(B.tile_entry, 0xff, 4ull * B.n_tiles, st);
  top_chain_kernel<<<1, 32, 0, st>>>(B.exit1, B.exit2, B.n, group_bytes, B.group_entry, B.result);
  tile_entry_kernel<<<cdiv(B.n_groups, 64), 64, 0, st>>>(B.exit1, B.group_entry, B.n, B.n_groups, group_bytes, B.tile_entry);
  cudaMemsetAsync(B.bitmap, 0, (size_t)B.n_tiles * (TILE / 8), st);
  tile_mark_thin_kernel<<<cdiv(B.n_tiles, 128), 128, 0, st>>>(B.step1, B.n_tiles, B.tile_entry, B.bitmap, B.tile_count);
  cudaMemsetAsync(B.tile_count + B.n_tiles, 0, 4, st);
  uint32_t launches = 5 + mscan(B.tile_count, B.tile_base, B.n_tiles + 1, 0, 1, B.scan_tmp, st);
  cudaMemcpyAsync(B.result + PARSE_R_NINS, B.tile_base + B.n_tiles, 4, cudaMemcpyDeviceToDevice, st);
  return launches;
}

void launch_parse_scatter(const ParseBounds& B, uint32_t* ins_pos, cudaStream_t st) {
  ins_scatter_kernel<<<B.n_tiles, TILE / 32, 0, st>>>(B.bitmap, B.tile_base, ins_pos);
}

uint32_t launch_parse_tree(const ParseTree& T, cudaStream_t st) {
  const uint32_t n1 = T.n_ins + 1;
  ins_info_kernel<<<cdiv(n1, 256), 256, 0, st>>>(T);
  uint32_t launches = 8;  // ins_info, heights, 3 x min64, link, shape, totals
  launches += mscan(T.delta, T.hb, n1, 0, 1, T.scan_tmp, st);
  heights_kernel<<<cdiv(n1, 256), 256, 0, st>>>(T);
  const uint32_t n_m1 = cdiv(n1, 64), n_m2 = cdiv(n_m1, 64), n_m3 = cdiv(n_m2, 64);
  min8_64_i16_kernel<<<cdiv(n_m1, 128), 128, 0, st>>>(T.h16, n1, T.m0, T.m1, n_m1);
  min64_i16_kernel<<<cdiv(n_m2, 128), 128, 0, st>>>(T.m1, n_m1, T.m2, n_m2);
  min64_i16_kernel<<<cdiv(n_m3, 128), 128, 0, st>>>(T.m2, n_m2, T.m3, n_m3);
  link_kernel16<<<cdiv(T.n_ins, 256), 256, 0, st>>>(T);
  shape_kernel<<<cdiv(n1, 256), 256, 0, st>>>(T);
  launches += mscan(T.cnt, T.scn, n1, T.cnt_stride, PARSE_N_CNT, T.scan_tmp, st);
  totals_kernel<<<1, 32, 0, st>>>(T);
  return launches;
}

void launch_parse_code_list(const ParseEmit& E, cudaStream_t st) { code_list_kernel<<<cdiv(E.T.n_ins, 256), 256, 0, st>>>(E); }

void launch_parse_emit(const ParseEmit& E, cudaStream_t st) {
  emit_kernel<<<cdiv(E.T.n_ins, 256), 256, 0, st>>>(E);
  if (E.n_keyed) emit_keyed_kernel<<<cdiv(E.n_keyed, 128), 128, 0, st>>>(E);
  climb_kernel<<<cdiv(E.T.n_ins, 256), 256, 0, st>>>(E);
}

}  // namespace ppd
