// encode.cuh — RLP / hex-prefix emitters that append straight into a thread's Keccak stage.
//
// Restates eth_trie_utils' node encoding (SURVEY.md 3.3 / row a18): hex-prefix keys, RLP strings
// and lists, child references (hash or raw RLP shorter than 32 bytes).  Everything is word-wise:
// byte strings at arbitrary global addresses are read as aligned 32-bit words and re-aligned with
// funnel shifts; a nibble-misaligned key suffix is shifted by four bits a word at a time.
#pragma once
#include <cstdint>

#include "keccak.cuh"

namespace ppd {
namespace enc {

__device__ __forceinline__ uint32_t len_prefix_size(uint32_t len) { return len < 56 ? 1 : len < 256 ? 2 : len < 65536 ? 3 : 4; }
// size of rlp_str(hex_prefix(nibbles)) for n nibbles: the one-byte case is always < 0x80
__device__ __forceinline__ uint32_t hex_prefix_str_size(uint32_t n) { return n < 2 ? 1 : 2 + (n >> 1); }

template <int B>
__device__ __forceinline__ void emit_len_prefix(Stage<B>& s, uint32_t len, uint32_t short_base, uint32_t long_base) {
  if (len < 56) {
    s.put_byte(short_base + len);
  } else if (len < 256) {
    s.put_partial((long_base + 1) | (len << 8), 2);
  } else if (len < 65536) {
    s.put_partial((long_base + 2) | ((len >> 8) << 8) | ((len & 255) << 16), 3);
  } else {
    s.put_partial((long_base + 3) | ((len >> 16) << 8) | (((len >> 8) & 255) << 16) | ((len & 255) << 24), 4);
  }
}

// cnt (1..4) bytes at an arbitrary global address as a little-endian word; touches only the aligned
// words that hold a requested byte
__device__ __forceinline__ uint32_t ld_bytes(const uint8_t* p, uint32_t cnt) {
  uintptr_t a = reinterpret_cast<uintptr_t>(p);
  const uint32_t* q = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  uint32_t ofs = (uint32_t)(a & 3);
  uint32_t lo = __ldg(q);
  uint32_t hi = (ofs + cnt > 4) ? __ldg(q + 1) : 0u;
  return __funnelshift_r(lo, hi, ofs * 8);
}

// n bytes that start at byte ofs (0..3) of aligned word 0 of a word source ld(i).  Branch-free in the
// alignment (lanes of a warp read values at different alignments): always the funnel-shift path, with
// the look-ahead load predicated on the word still holding a requested byte.
template <int B, class Ld>
__device__ __forceinline__ void emit_words(Stage<B>& s, const Ld& ld, uint32_t ofs, uint32_t n) {
  if (n == 0) return;
  const uint32_t sh = ofs * 8;
  const uint32_t nwords = (ofs + n + 3) >> 2;  // aligned words that hold a requested byte
  const uint32_t full = n >> 2, rem = n & 3;
  uint32_t cur = ld(0u);
  for (uint32_t i = 0; i < full; i++) {
    uint32_t nxt = (i + 1 < nwords) ? ld(i + 1) : 0u;
    s.put_word(__funnelshift_r(cur, nxt, sh));
    cur = nxt;
  }
  if (rem) {
    uint32_t nxt = (full + 1 < nwords) ? ld(full + 1) : 0u;
    s.put_partial(__funnelshift_r(cur, nxt, sh), rem);
  }
}
// n bytes from any global address
template <int B>
__device__ __forceinline__ void emit_bytes(Stage<B>& s, const uint8_t* p, uint32_t n) {
  uintptr_t a = reinterpret_cast<uintptr_t>(p);
  const uint32_t* q = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  emit_words(s, [q](uint32_t i) { return __ldg(q + i); }, (uint32_t)(a & 3), n);
}

// m bytes of a packed nibble string that starts at the high (odd == 0) or the low (odd == 1)
// nibble of p[0]:  odd == 0: out[k] = in[k];  odd == 1: out[k] = (in[k] & 15) << 4 | in[k + 1] >> 4.
// Branch-free in `odd` (lanes of a warp sit at depths of both parities).
template <int B>
__device__ __forceinline__ void emit_nibble_bytes(Stage<B>& s, const uint8_t* p, uint32_t m, uint32_t odd) {
  const uint32_t avail = m + odd;  // bytes readable from p
  uint32_t k = 0;
  uint32_t W = ld_bytes(p, min(4u, avail));
  while (m - k >= 4) {
    uint32_t left = avail - (k + 4);
    uint32_t Wn = left ? ld_bytes(p + k + 4, min(4u, left)) : 0u;
    uint32_t W1 = __funnelshift_r(W, Wn, 8);
    uint32_t shifted = ((W & 0x0f0f0f0fu) << 4) | ((W1 >> 4) & 0x0f0f0f0fu);
    s.put_word(odd ? shifted : W);
    W = Wn;
    k += 4;
  }
  uint32_t r = m - k;
  if (r) {
    uint32_t shifted = ((W & 0x0f0f0f0fu) << 4) | ((W >> 12) & 0x0f0f0f0fu);
    s.put_partial(odd ? shifted : W, r);
  }
}

// rlp_str(hex_prefix(nibbles [start, start + n) of the packed key, is_leaf)): at most 34 bytes
template <int B>
__device__ __forceinline__ void emit_hex_prefix_str(Stage<B>& s, const uint8_t* key, uint32_t start, uint32_t n, uint32_t is_leaf) {
  if (n >= 2) s.put_byte(0x80 + 1 + (n >> 1));
  const uint32_t flag = (is_leaf ? 2u : 0u) + (n & 1);
  uint32_t first = flag << 4;
  if (n & 1) {
    uint32_t b = __ldg(key + (start >> 1));
    first |= (start & 1) ? (b & 15) : (b >> 4);
  }
  s.put_byte(first);
  const uint32_t j = start + (n & 1), m = n >> 1;
  if (m) emit_nibble_bytes(s, key + (j >> 1), m, j & 1);
}

// a child reference inside a parent: 0xa0 || hash, or the child's raw RLP when shorter than 32 bytes
template <int B>
__device__ __forceinline__ void emit_ref(Stage<B>& s, const uint4& x, const uint4& y, uint32_t len) {
  if (len == 32) {
    s.put_byte(0xa0);
    s.put_word(x.x), s.put_word(x.y), s.put_word(x.z), s.put_word(x.w);
    s.put_word(y.x), s.put_word(y.y), s.put_word(y.z), s.put_word(y.w);
  } else {
    uint32_t w[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
#pragma unroll
    for (int i = 0; i < 8; i++) {
      uint32_t take = len > 4u * i ? min(4u, len - 4u * i) : 0u;
      s.put_partial(w[i], take);
    }
  }
}
template <int B>
__device__ __forceinline__ void emit_ref_at(Stage<B>& s, const uint8_t* ref32, uint32_t len) {
  const uint4* q = reinterpret_cast<const uint4*>(ref32);
  uint4 x = __ldcg(q), y = __ldcg(q + 1);
  emit_ref(s, x, y, len);
}

// significant bytes of a big-endian U256 stored in 32 bytes (4-byte aligned)
__device__ __forceinline__ uint32_t u256_sig_bytes(const uint8_t* be32) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(be32);
  uint32_t lead = 32;
#pragma unroll
  for (int i = 7; i >= 0; i--) {
    uint32_t v = __byte_perm(__ldg(w + i), 0, 0x0123);  // big-endian value of bytes 4i .. 4i+3
    if (v) lead = 4u * i + (__clz(v) >> 3);
  }
  return 32 - lead;
}
__device__ __forceinline__ uint32_t u256_str_size(const uint8_t* be32, uint32_t nbytes) {
  if (nbytes == 0) return 1;
  if (nbytes == 1 && __ldg(be32 + 31) < 0x80) return 1;
  return 1 + nbytes;
}
// rlp of a U256 as a minimal big-endian string: at most 33 bytes
template <int B>
__device__ __forceinline__ void emit_u256_str(Stage<B>& s, const uint8_t* be32, uint32_t nbytes) {
  if (nbytes == 0) {
    s.put_byte(0x80);
    return;
  }
  if (!(nbytes == 1 && __ldg(be32 + 31) < 0x80)) s.put_byte(0x80 + nbytes);
  emit_bytes(s, be32 + 32 - nbytes, nbytes);
}

__device__ __forceinline__ void digest_words(const uint64_t (&a)[25], uint4& x, uint4& y) {
  x = make_uint4((uint32_t)a[0], (uint32_t)(a[0] >> 32), (uint32_t)a[1], (uint32_t)(a[1] >> 32));
  y = make_uint4((uint32_t)a[2], (uint32_t)(a[2] >> 32), (uint32_t)a[3], (uint32_t)(a[3] >> 32));
}

// the first `total` (< 32) bytes of the stage's current block as a zero-padded 32-byte ref
template <int B>
__device__ __forceinline__ void inline_ref_words(Stage<B>& s, uint32_t total, uint4& x, uint4& y) {
  s.flush_partial();
  uint32_t h[8] = {s.template word<0>(), s.template word<1>(), s.template word<2>(), s.template word<3>(),
                   s.template word<4>(), s.template word<5>(), s.template word<6>(), s.template word<7>()};
  // word k keeps its first total - 4k bytes (a mask per word: a test against the last word's index lets the
  // compiler turn the loop into a store to h[nw - 1], which puts h in local memory)
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const int rem = (int)total - 4 * k;
    h[k] &= rem >= 4 ? 0xffffffffu : rem > 0 ? (1u << (8 * rem)) - 1 : 0u;
  }
  x = make_uint4(h[0], h[1], h[2], h[3]);
  y = make_uint4(h[4], h[5], h[6], h[7]);
}

// g bytes of 0x80 (empty branch slots / the empty branch value), g <= 17
template <int B>
__device__ __forceinline__ void emit_empty_run(Stage<B>& s, uint32_t g) {
  while (g >= 4) {
    s.put_word(0x80808080u);
    g -= 4;
  }
  s.put_partial(0x80808080u, g);
}

// per-warp accumulation of the work counters: one atomic triple per warp
__device__ __forceinline__ void add_counters(unsigned long long* counters, uint32_t hashed, uint32_t perms, uint32_t enc_bytes) {
  if (!counters) return;
  for (int off = 16; off > 0; off >>= 1) {
    hashed += __shfl_down_sync(0xffffffffu, hashed, off);
    perms += __shfl_down_sync(0xffffffffu, perms, off);
    enc_bytes += __shfl_down_sync(0xffffffffu, enc_bytes, off);
  }
  if ((threadIdx.x & 31) == 0 && hashed) {
    atomicAdd(counters + 0, (unsigned long long)hashed);
    atomicAdd(counters + 1, (unsigned long long)perms);
    atomicAdd(counters + 2, (unsigned long long)enc_bytes);
  }
}

}  // namespace enc
}  // namespace ppd
