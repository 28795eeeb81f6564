// ppd_leaves.cu — leaves in any order, with repeated and optionally unhashed keys, turned into the strictly ascending,
// de-duplicated leaves that the builder of ppd_build.cu takes (ppd_trie_root_leaves[_dev], DESIGN.md §6).
//
// The reference builds a trie by inserting leaf after leaf (eth_trie_utils `insert`; compact_to_partial_trie.rs:105,125):
// keys come in any order and a repeated key keeps the value of its last insertion.  Here:
//   hash_fixed_keys_kernel   keccak256 of n keys of one length (PPD_LEAVES_HASH_KEYS): one rate block each
//   key_word_kernel          big-endian 64-bit word w of every key, paired with its input position
//   digit_counts_kernel      counts of the 8 byte digits of n 64-bit keys: a digit of one value skips its pass
//   radix_tile_hist_kernel   one pass of a stable LSD radix sort of (u64 key, u32 value) pairs: per-tile digit counts,
//   radix_scatter_kernel     exclusive_scan of them (digit-major), and a scatter with in-tile ranks
//   tie_*_kernel             positions equal to their predecessor on the words sorted so far; the tied runs are
//                            compacted, re-sorted on the next word (then stably by run) and written back
//   keep_kernel / gather_kernel   the last element of every run of equal keys, packed with its value
#include <cstdint>

#include "encode.cuh"
#include "keccak.cuh"
#include "ppd_kernels.h"

namespace ppd {

using namespace enc;
static constexpr uint32_t FULL = 0xffffffffu;

// ------------------------------------------------------------------ input checks / key hashing -------

// flag |= 1 when val_off decreases anywhere or val_off[n] > vals_bytes
__global__ void check_offsets_kernel(const uint64_t* __restrict__ off, uint32_t n, uint64_t vals_bytes, uint32_t* __restrict__ flag) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t a = off[i], b = off[i + 1];
  if (a > b || (i == n - 1 && b > vals_bytes)) atomicOr(flag, 1u);
}

// key i = keys[i * key_len .. + key_len), key_len <= 135: one padded rate block, one permutation (the sponge of
// keccak256_batch_kernel, with the offsets implied by the fixed stride)
template <int B>
__global__ void __launch_bounds__(B) hash_fixed_keys_kernel(const uint8_t* __restrict__ keys, uint32_t key_len, uint32_t n, uint8_t* __restrict__ out) {
  __shared__ uint32_t smem[PPD_STAGE_WORDS * B];
  const uint32_t i = blockIdx.x * B + threadIdx.x;
  if (blockIdx.x * B >= n) return;  // (block-uniform)
  Stage<B> s;
  s.init(smem);
  uint64_t a[25];
#pragma unroll
  for (int k = 0; k < 25; k++) a[k] = 0;
  if (i < n) emit_bytes(s, keys + (uint64_t)i * key_len, key_len);
  s.pad();
  absorb_stage<B>(a, s);
  keccak_f1600(a);
  if (i < n) {
    uint4 x, y;
    digest_words(a, x, y);
    uint4* o = reinterpret_cast<uint4*>(out + 32ull * i);
    o[0] = x, o[1] = y;
  }
}

// big-endian 64-bit word w of the 32-byte key at p (any alignment)
__device__ __forceinline__ uint64_t key_word(const uint8_t* p, int w) {
  p += 8 * w;
  if ((reinterpret_cast<uintptr_t>(p) & 7) == 0) {
    const uint2 x = __ldg(reinterpret_cast<const uint2*>(p));
    return (uint64_t)__byte_perm(x.x, 0, 0x0123) << 32 | __byte_perm(x.y, 0, 0x0123);
  }
  uint64_t v = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) v = v << 8 | __ldg(p + k);
  return v;
}

// out_key[i] = word w of key i; out_val[i] = i
__global__ void key_word_kernel(const uint8_t* __restrict__ keys32, uint32_t n, int w, uint64_t* __restrict__ out_key, uint32_t* __restrict__ out_val) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out_key[i] = key_word(keys32 + 32ull * i, w);
  out_val[i] = i;
}

// counts[8 * 256]: counts[256 * p + d] = number of keys whose byte digit p (bits 8p .. 8p + 7) is d
__global__ void __launch_bounds__(256) digit_counts_kernel(const uint64_t* __restrict__ keys, uint32_t n, uint32_t* __restrict__ counts) {
  __shared__ uint32_t h[8 * 256];
  for (uint32_t j = threadIdx.x; j < 8 * 256; j += 256) h[j] = 0;
  __syncthreads();
  for (uint32_t i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
    uint64_t k = keys[i];
#pragma unroll
    for (int p = 0; p < 8; p++) atomicAdd(&h[256 * p + ((k >> (8 * p)) & 255)], 1u);
  }
  __syncthreads();
  for (uint32_t j = threadIdx.x; j < 8 * 256; j += 256)
    if (h[j]) atomicAdd(&counts[j], h[j]);
}

// ------------------------------------------------------------------ one radix pass -------
// A tile is RADIX_TILE consecutive elements; warp w of the scatter owns RADIX_ITEMS chunks of 32 consecutive elements
// in a row.  hist[d * n_tiles + t] = elements of tile t with digit d, so that its exclusive scan is the first output
// position of (digit d, tile t).
static constexpr int RADIX_B = 256, RADIX_ITEMS = 16, RADIX_WARPS = RADIX_B / 32;
static constexpr uint32_t RADIX_TILE = RADIX_B * RADIX_ITEMS;  // 4096

__global__ void __launch_bounds__(RADIX_B) radix_tile_hist_kernel(const uint64_t* __restrict__ keys, uint32_t n, int shift, uint32_t n_tiles,
                                                                  uint32_t* __restrict__ hist) {
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t base = (uint64_t)blockIdx.x * RADIX_TILE + threadIdx.x;
#pragma unroll
  for (int k = 0; k < RADIX_ITEMS; k++) {
    uint64_t e = base + k * RADIX_B;
    if (e < n) atomicAdd(&h[(keys[e] >> shift) & 255], 1u);
  }
  __syncthreads();
  hist[(uint64_t)threadIdx.x * n_tiles + blockIdx.x] = h[threadIdx.x];
}

// Stable: inside a tile, an element's rank among the elements of its digit is the number of them before it (earlier
// chunks of its warp through the warp's running counters, earlier warps through the per-digit scan over warps,
// earlier lanes of its chunk through the match mask).
__global__ void __launch_bounds__(RADIX_B) radix_scatter_kernel(const uint64_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                                                                uint64_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, uint32_t n,
                                                                int shift, uint32_t n_tiles, const uint32_t* __restrict__ hist_scan) {
  __shared__ uint32_t cnt[RADIX_WARPS * 256];
  const uint32_t lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t* my = cnt + 256 * w;
  for (uint32_t j = lane; j < 256; j += 32) my[j] = 0;
  __syncwarp();
  const uint32_t lt = (1u << lane) - 1;
  const uint64_t e0 = (uint64_t)blockIdx.x * RADIX_TILE + (uint64_t)w * (32 * RADIX_ITEMS) + lane;
  uint64_t key[RADIX_ITEMS];
  uint32_t val[RADIX_ITEMS], rank[RADIX_ITEMS];
#pragma unroll
  for (int k = 0; k < RADIX_ITEMS; k++) {
    const uint64_t e = e0 + 32 * k;
    key[k] = e < n ? keys_in[e] : 0;
    val[k] = e < n ? vals_in[e] : 0;
  }
#pragma unroll
  for (int k = 0; k < RADIX_ITEMS; k++) {
    const bool valid = e0 + 32 * k < n;
    const uint32_t d = valid ? (uint32_t)(key[k] >> shift) & 255 : 256u;
    const uint32_t peers = __match_any_sync(FULL, d);
    const uint32_t before = valid ? my[d] : 0u;
    __syncwarp();
    if (valid && (peers & lt) == 0) my[d] = before + __popc(peers);
    __syncwarp();
    rank[k] = before + __popc(peers & lt);
  }
  __syncthreads();
  {
    const uint32_t d = threadIdx.x;  // RADIX_B == 256 digits
    uint32_t run = hist_scan[(uint64_t)d * n_tiles + blockIdx.x];
#pragma unroll
    for (int v = 0; v < RADIX_WARPS; v++) {
      uint32_t c = cnt[256 * v + d];
      cnt[256 * v + d] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < RADIX_ITEMS; k++) {
    if (e0 + 32 * k < n) {
      const uint32_t dst = my[(uint32_t)(key[k] >> shift) & 255] + rank[k];
      keys_out[dst] = key[k];
      vals_out[dst] = val[k];
    }
  }
}

// ------------------------------------------------------------------ ties -------

// tie[i] = (i > 0 && k[i] == k[i - 1]), tie[n] = 0; *count += number of ties
__global__ void tie_flags_kernel(const uint64_t* __restrict__ k, uint32_t n, uint32_t* __restrict__ tie, uint32_t* __restrict__ count) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  bool t = i > 0 && i < n && k[i] == k[i - 1];
  if (i <= n) tie[i] = t;
  uint32_t c = __syncthreads_count(t);
  if (threadIdx.x == 0 && c) atomicAdd(count, c);
}

// member[i]: i is in a run of tied elements; start[i]: i is its first element (entry n of both: 0)
__global__ void tie_members_kernel(const uint32_t* __restrict__ tie, uint32_t n, uint32_t* __restrict__ member, uint32_t* __restrict__ start) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  uint32_t t0 = i < n ? tie[i] : 0u, t1 = i + 1 < n ? tie[i + 1] : 0u;
  uint32_t m = t0 | t1;
  member[i] = m;
  start[i] = m & (t0 ^ 1u);
}

// the members, compacted in order: their position, input index, run, word w of their key; key/val: what sort A orders
__global__ void tie_compact_kernel(const uint8_t* __restrict__ keys32, const uint32_t* __restrict__ idx, uint32_t n, int w,
                                   const uint32_t* __restrict__ member, const uint32_t* __restrict__ mpos, const uint32_t* __restrict__ start,
                                   const uint32_t* __restrict__ spos, uint32_t* __restrict__ cpos, uint32_t* __restrict__ cidx,
                                   uint32_t* __restrict__ crun, uint64_t* __restrict__ cword, uint64_t* __restrict__ key, uint32_t* __restrict__ val) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !member[i]) return;
  const uint32_t j = mpos[i], s = idx[i];
  const uint64_t word = key_word(keys32 + 32ull * s, w);
  cpos[j] = i;
  cidx[j] = s;
  crun[j] = spos[i] + start[i] - 1;
  cword[j] = word;
  key[j] = word;
  val[j] = j;
}

// sort B's input: the run of each member in sort A's order
__global__ void tie_run_key_kernel(const uint32_t* __restrict__ crun, const uint32_t* __restrict__ order, uint32_t m, uint64_t* __restrict__ key,
                                   uint32_t* __restrict__ val) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  uint32_t j = order[t];
  key[t] = crun[j];
  val[t] = j;
}

// the t-th member in (run, word, previous order) order goes to the t-th member position: a run keeps its positions
__global__ void tie_writeback_kernel(const uint32_t* __restrict__ cpos, const uint32_t* __restrict__ cidx, const uint32_t* __restrict__ crun,
                                     const uint64_t* __restrict__ cword, const uint32_t* __restrict__ order, uint32_t m, uint32_t* __restrict__ idx,
                                     uint32_t* __restrict__ tie, uint32_t* __restrict__ count) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  bool tied = false;
  if (t < m) {
    const uint32_t j = order[t], i = cpos[t];
    idx[i] = cidx[j];
    if (t > 0) {
      const uint32_t p = order[t - 1];
      tied = crun[p] == crun[j] && cword[p] == cword[j];
    }
    tie[i] = tied;
  }
  uint32_t c = __syncthreads_count(tied);
  if (threadIdx.x == 0 && c) atomicAdd(count, c);
}

// ------------------------------------------------------------------ keep the last, gather -------

// the sort is stable in input position, so the last element of a run of equal keys is the key's last occurrence
__global__ void keep_kernel(const uint32_t* __restrict__ tie, const uint32_t* __restrict__ idx, const uint64_t* __restrict__ val_off, uint32_t n,
                            uint32_t* __restrict__ keep, uint64_t* __restrict__ len) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  uint32_t k = i < n && (i + 1 == n || !tie[i + 1]);
  keep[i] = k;
  uint64_t l = 0;
  if (k) {
    uint32_t s = idx[i];
    l = val_off[s + 1] - val_off[s];
  }
  len[i] = l;
}

// n bytes from src (any alignment) to dst (any alignment): 32-bit stores once dst is aligned, each assembled from
// the two aligned source words it straddles
__device__ __forceinline__ void copy_bytes(uint8_t* dst, const uint8_t* src, uint64_t n) {
  while (n && (reinterpret_cast<uintptr_t>(dst) & 3)) {
    *dst++ = __ldg(src++);
    n--;
  }
  const uintptr_t a = reinterpret_cast<uintptr_t>(src);
  const uint32_t* q = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3) * 8;
  uint32_t* d = reinterpret_cast<uint32_t*>(dst);
  const uint64_t words = n >> 2;
  for (uint64_t k = 0; k < words; k++) {
    uint32_t lo = __ldg(q + k), hi = sh ? __ldg(q + k + 1) : 0u;
    d[k] = __funnelshift_r(lo, hi, sh);
  }
  dst += 4 * words, src += 4 * words;
  for (uint32_t r = (uint32_t)(n & 3); r; r--) *dst++ = __ldg(src++);
}

__global__ void gather_kernel(const uint8_t* __restrict__ keys32, const uint32_t* __restrict__ idx, const uint64_t* __restrict__ val_off,
                              const uint8_t* __restrict__ vals, uint32_t n, const uint32_t* __restrict__ keep, const uint32_t* __restrict__ kpos,
                              const uint64_t* __restrict__ koff, uint8_t* __restrict__ keys_out, uint64_t* __restrict__ off_out,
                              uint8_t* __restrict__ vals_out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) {
    off_out[kpos[n]] = koff[n];
    return;
  }
  if (!keep[i]) return;
  const uint32_t j = kpos[i], s = idx[i];
  const uint8_t* kp = keys32 + 32ull * s;
  uint4* ko = reinterpret_cast<uint4*>(keys_out + 32ull * j);
  if ((reinterpret_cast<uintptr_t>(kp) & 15) == 0) {
    ko[0] = __ldg(reinterpret_cast<const uint4*>(kp)), ko[1] = __ldg(reinterpret_cast<const uint4*>(kp) + 1);
  } else {
    copy_bytes(keys_out + 32ull * j, kp, 32);
  }
  const uint64_t o = koff[i];
  off_out[j] = o;
  const uint64_t b = val_off[s];
  copy_bytes(vals_out + o, vals + b, val_off[s + 1] - b);
}

// ------------------------------------------------------------------ launchers -------
static inline uint32_t grid(uint64_t n, uint32_t b) { return (uint32_t)((n + b - 1) / b); }

void launch_check_offsets(const uint64_t* val_off, uint32_t n, uint64_t vals_bytes, uint32_t* flag, cudaStream_t st) {
  check_offsets_kernel<<<grid(n, 256), 256, 0, st>>>(val_off, n, vals_bytes, flag);
}
static constexpr int HK_B = 128;
void launch_hash_fixed_keys(const uint8_t* keys, uint32_t key_len, uint32_t n, uint8_t* out32, cudaStream_t st) {
  hash_fixed_keys_kernel<HK_B><<<grid(n, HK_B), HK_B, 0, st>>>(keys, key_len, n, out32);
}
void launch_key_word(const uint8_t* keys32, uint32_t n, int w, uint64_t* out_key, uint32_t* out_val, cudaStream_t st) {
  key_word_kernel<<<grid(n, 256), 256, 0, st>>>(keys32, n, w, out_key, out_val);
}
void launch_digit_counts(const uint64_t* keys, uint32_t n, uint32_t* counts, cudaStream_t st) {
  uint32_t g = grid(n, 256 * 16);
  digit_counts_kernel<<<g < 2048 ? g : 2048, 256, 0, st>>>(keys, n, counts);
}
size_t radix_hist_words(uint32_t n) { return 256ull * grid(n, RADIX_TILE); }
uint32_t launch_radix_pass(const uint64_t* keys_in, const uint32_t* vals_in, uint64_t* keys_out, uint32_t* vals_out, uint32_t n, int digit,
                           uint32_t* hist, uint32_t* hist_scan, uint32_t* scan_tmp, cudaStream_t st) {
  const uint32_t tiles = grid(n, RADIX_TILE);
  radix_tile_hist_kernel<<<tiles, RADIX_B, 0, st>>>(keys_in, n, 8 * digit, tiles, hist);
  const uint32_t scans = exclusive_scan(hist, hist_scan, 256 * tiles, scan_tmp, st);
  radix_scatter_kernel<<<tiles, RADIX_B, 0, st>>>(keys_in, vals_in, keys_out, vals_out, n, 8 * digit, tiles, hist_scan);
  return 2 + scans;
}
void launch_tie_flags(const uint64_t* sorted_keys, uint32_t n, uint32_t* tie, uint32_t* count, cudaStream_t st) {
  tie_flags_kernel<<<grid(n + 1, 256), 256, 0, st>>>(sorted_keys, n, tie, count);
}
void launch_tie_members(const uint32_t* tie, uint32_t n, uint32_t* member, uint32_t* start, cudaStream_t st) {
  tie_members_kernel<<<grid(n + 1, 256), 256, 0, st>>>(tie, n, member, start);
}
void launch_tie_compact(const TieRuns& R, const uint8_t* keys32, const uint32_t* idx, uint32_t n, int w, uint64_t* key, uint32_t* val,
                        cudaStream_t st) {
  tie_compact_kernel<<<grid(n, 256), 256, 0, st>>>(keys32, idx, n, w, R.member, R.mpos, R.start, R.spos, R.cpos, R.cidx, R.crun, R.cword, key, val);
}
void launch_tie_run_key(const TieRuns& R, const uint32_t* order, uint32_t m, uint64_t* key, uint32_t* val, cudaStream_t st) {
  if (m) tie_run_key_kernel<<<grid(m, 256), 256, 0, st>>>(R.crun, order, m, key, val);
}
void launch_tie_writeback(const TieRuns& R, const uint32_t* order, uint32_t m, uint32_t* idx, uint32_t* tie, uint32_t* count, cudaStream_t st) {
  if (m) tie_writeback_kernel<<<grid(m, 256), 256, 0, st>>>(R.cpos, R.cidx, R.crun, R.cword, order, m, idx, tie, count);
}
void launch_keep_last(const uint32_t* tie, const uint32_t* idx, const uint64_t* val_off, uint32_t n, uint32_t* keep, uint64_t* len, cudaStream_t st) {
  keep_kernel<<<grid(n + 1, 256), 256, 0, st>>>(tie, idx, val_off, n, keep, len);
}
void launch_gather_leaves(const uint8_t* keys32, const uint32_t* idx, const uint64_t* val_off, const uint8_t* vals, uint32_t n, const uint32_t* keep,
                          const uint32_t* kpos, const uint64_t* koff, uint8_t* keys_out, uint64_t* off_out, uint8_t* vals_out, cudaStream_t st) {
  gather_kernel<<<grid(n + 1, 256), 256, 0, st>>>(keys32, idx, val_off, vals, n, keep, kpos, koff, keys_out, off_out, vals_out);
}

}  // namespace ppd
