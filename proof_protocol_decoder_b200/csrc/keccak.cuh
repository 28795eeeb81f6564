// keccak.cuh — Keccak-256 for sm_100a, thread-per-sponge.
//
// Replaces: keccak-hash 0.10.0 -> tiny-keccak 2.0.2 as called through
// protocol_decoder/src/utils.rs:11-13 (`hash`) and, for trie nodes, eth_trie_utils'
// `hash_bytes_if_large_enough` (SURVEY.md 3.3 / row a18).
//
// Layout: the 25 x 64-bit state lives in registers as 32-bit halves.  Per round on the 32-bit
// ISA: theta = 20 LOP3 (5-input column parities) + 10 SHF (rotl1) + 50 LOP3 (3-input XOR applying
// D), rho = 48 SHF, pi = register renaming, chi = 50 LOP3 (a ^ (~b & c)), iota <= 2: ~180
// ALU-pipe instructions per round, 4 320 per permutation (DESIGN.md "Keccak roofline").
#pragma once
#include <cstdint>

namespace ppd {

__constant__ uint64_t KECCAK_RC[24] = {
    0x0000000000000001ULL, 0x0000000000008082ULL, 0x800000000000808aULL, 0x8000000080008000ULL,
    0x000000000000808bULL, 0x0000000080000001ULL, 0x8000000080008081ULL, 0x8000000000008009ULL,
    0x000000000000008aULL, 0x0000000000000088ULL, 0x0000000080008009ULL, 0x000000008000000aULL,
    0x000000008000808bULL, 0x800000000000008bULL, 0x8000000000008089ULL, 0x8000000000008003ULL,
    0x8000000000008002ULL, 0x8000000000000080ULL, 0x000000000000800aULL, 0x800000008000000aULL,
    0x8000000080008081ULL, 0x8000000000008080ULL, 0x0000000080000001ULL, 0x8000000080008008ULL};

// Multipliers 2^k in constant memory: ptxas cannot strength-reduce a multiply by c[bank] into a
// shift, so rotl64_mad below really issues on the FMA pipe (IMAD.WIDE) instead of the ALU pipe.
__constant__ uint32_t KECCAK_POW2[32] = {1u << 0,  1u << 1,  1u << 2,  1u << 3,  1u << 4,  1u << 5,  1u << 6,  1u << 7,
                                         1u << 8,  1u << 9,  1u << 10, 1u << 11, 1u << 12, 1u << 13, 1u << 14, 1u << 15,
                                         1u << 16, 1u << 17, 1u << 18, 1u << 19, 1u << 20, 1u << 21, 1u << 22, 1u << 23,
                                         1u << 24, 1u << 25, 1u << 26, 1u << 27, 1u << 28, 1u << 29, 1u << 30, 1u << 31};

// 64-bit rotate-left entirely on the FMA pipe (no LOP3/SHF):
//   t = lo * 2^k  (IMAD.WIDE)  -> t.hi = lo >> (32-k)        new_hi = hi * 2^k + t.hi   (IMAD)
//   u = hi * 2^k  (IMAD.WIDE)  -> u.hi = hi >> (32-k)        new_lo = lo * 2^k + u.hi   (IMAD)
// (the two addends never overlap, so + is |).  4 FMA-pipe instructions instead of 2 ALU-pipe ones.
template <int K>
__device__ __forceinline__ uint64_t rotl64_mad(uint64_t x) {
  static_assert(K > 0 && K < 64 && K != 32, "rotation amount");
  uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
  if (K > 32) {
    uint32_t t = lo;
    lo = hi;
    hi = t;
  }
  const uint32_t m = KECCAK_POW2[K & 31];
  uint64_t t, u;
  uint32_t nlo, nhi;
  asm("mul.wide.u32 %0, %1, %2;" : "=l"(t) : "r"(lo), "r"(m));
  asm("mul.wide.u32 %0, %1, %2;" : "=l"(u) : "r"(hi), "r"(m));
  asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(nhi) : "r"(hi), "r"(m), "r"((uint32_t)(t >> 32)));
  asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(nlo) : "r"(lo), "r"(m), "r"((uint32_t)(u >> 32)));
  return ((uint64_t)nhi << 32) | nlo;
}

// 64-bit rotate-left by a compile-time amount as two funnel shifts on the halves
template <int K>
__device__ __forceinline__ uint64_t rotl64(uint64_t x) {
  static_assert(K > 0 && K < 64, "rotation amount");
  uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
  uint32_t nlo, nhi;
  if (K < 32) {
    nhi = __funnelshift_l(lo, hi, (uint32_t)K);
    nlo = __funnelshift_l(hi, lo, (uint32_t)K);
  } else if (K == 32) {
    nhi = lo;
    nlo = hi;
  } else {
    nhi = __funnelshift_l(hi, lo, (uint32_t)(K - 32));
    nlo = __funnelshift_l(lo, hi, (uint32_t)(K - 32));
  }
  return ((uint64_t)nhi << 32) | nlo;
}

__device__ __forceinline__ uint64_t xor3(uint64_t a, uint64_t b, uint64_t c) {
  uint32_t lo, hi;
  asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(lo) : "r"((uint32_t)a), "r"((uint32_t)b), "r"((uint32_t)c));
  asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(hi) : "r"((uint32_t)(a >> 32)), "r"((uint32_t)(b >> 32)), "r"((uint32_t)(c >> 32)));
  return ((uint64_t)hi << 32) | lo;
}
// a ^ (~b & c)
__device__ __forceinline__ uint64_t chi1(uint64_t a, uint64_t b, uint64_t c) {
  uint32_t lo, hi;
  asm("lop3.b32 %0, %1, %2, %3, 0xD2;" : "=r"(lo) : "r"((uint32_t)a), "r"((uint32_t)b), "r"((uint32_t)c));
  asm("lop3.b32 %0, %1, %2, %3, 0xD2;" : "=r"(hi) : "r"((uint32_t)(a >> 32)), "r"((uint32_t)(b >> 32)), "r"((uint32_t)(c >> 32)));
  return ((uint64_t)hi << 32) | lo;
}

// rho rotation of lane I: on the FMA pipe for the lanes selected by MAD_MASK, else on the ALU pipe
template <int K, int I, uint32_t MAD_MASK>
__device__ __forceinline__ uint64_t rho(uint64_t x) {
  if constexpr (((MAD_MASK >> I) & 1u) != 0 && K != 32)
    return rotl64_mad<K>(x);
  else
    return rotl64<K>(x);
}

// One round.  Reads a[], writes a[] (through a register-renamed b[]).
template <uint32_t MAD_MASK>
__device__ __forceinline__ void keccak_round(uint64_t (&a)[25], uint64_t rc) {
  uint64_t c0 = xor3(xor3(a[0], a[5], a[10]), a[15], a[20]);
  uint64_t c1 = xor3(xor3(a[1], a[6], a[11]), a[16], a[21]);
  uint64_t c2 = xor3(xor3(a[2], a[7], a[12]), a[17], a[22]);
  uint64_t c3 = xor3(xor3(a[3], a[8], a[13]), a[18], a[23]);
  uint64_t c4 = xor3(xor3(a[4], a[9], a[14]), a[19], a[24]);
  uint64_t r0 = rotl64<1>(c0), r1 = rotl64<1>(c1), r2 = rotl64<1>(c2), r3 = rotl64<1>(c3), r4 = rotl64<1>(c4);
  // theta folded into the rho/pi gather: t = a ^ c[x-1] ^ rotl1(c[x+1]) is one LOP3 per half
  uint64_t b[25];
#define TH(i, x) xor3(a[i], (x == 0 ? c4 : x == 1 ? c0 : x == 2 ? c1 : x == 3 ? c2 : c3), (x == 0 ? r1 : x == 1 ? r2 : x == 2 ? r3 : x == 3 ? r4 : r0))
  b[0] = TH(0, 0);
  b[10] = rho<1, 1, MAD_MASK>(TH(1, 1));
  b[20] = rho<62, 2, MAD_MASK>(TH(2, 2));
  b[5] = rho<28, 3, MAD_MASK>(TH(3, 3));
  b[15] = rho<27, 4, MAD_MASK>(TH(4, 4));
  b[16] = rho<36, 5, MAD_MASK>(TH(5, 0));
  b[1] = rho<44, 6, MAD_MASK>(TH(6, 1));
  b[11] = rho<6, 7, MAD_MASK>(TH(7, 2));
  b[21] = rho<55, 8, MAD_MASK>(TH(8, 3));
  b[6] = rho<20, 9, MAD_MASK>(TH(9, 4));
  b[7] = rho<3, 10, MAD_MASK>(TH(10, 0));
  b[17] = rho<10, 11, MAD_MASK>(TH(11, 1));
  b[2] = rho<43, 12, MAD_MASK>(TH(12, 2));
  b[12] = rho<25, 13, MAD_MASK>(TH(13, 3));
  b[22] = rho<39, 14, MAD_MASK>(TH(14, 4));
  b[23] = rho<41, 15, MAD_MASK>(TH(15, 0));
  b[8] = rho<45, 16, MAD_MASK>(TH(16, 1));
  b[18] = rho<15, 17, MAD_MASK>(TH(17, 2));
  b[3] = rho<21, 18, MAD_MASK>(TH(18, 3));
  b[13] = rho<8, 19, MAD_MASK>(TH(19, 4));
  b[14] = rho<18, 20, MAD_MASK>(TH(20, 0));
  b[24] = rho<2, 21, MAD_MASK>(TH(21, 1));
  b[9] = rho<61, 22, MAD_MASK>(TH(22, 2));
  b[19] = rho<56, 23, MAD_MASK>(TH(23, 3));
  b[4] = rho<14, 24, MAD_MASK>(TH(24, 4));
#undef TH
#pragma unroll
  for (int y = 0; y < 25; y += 5) {
    a[y + 0] = chi1(b[y + 0], b[y + 1], b[y + 2]);
    a[y + 1] = chi1(b[y + 1], b[y + 2], b[y + 3]);
    a[y + 2] = chi1(b[y + 2], b[y + 3], b[y + 4]);
    a[y + 3] = chi1(b[y + 3], b[y + 4], b[y + 0]);
    a[y + 4] = chi1(b[y + 4], b[y + 0], b[y + 1]);
  }
  a[0] ^= rc;
}

#ifndef PPD_KECCAK_UNROLL
#define PPD_KECCAK_UNROLL 2
#endif
#define PPD_PRAGMA_(x) _Pragma(#x)
#define PPD_PRAGMA_UNROLL(n) PPD_PRAGMA_(unroll n)

#ifndef PPD_KECCAK_MAD_MASK
#define PPD_KECCAK_MAD_MASK 0u
#endif

template <int UNROLL, uint32_t MAD_MASK>
__device__ __forceinline__ void keccak_f1600_t(uint64_t (&a)[25]) {
  if constexpr (UNROLL >= 24) {
#pragma unroll
    for (int r = 0; r < 24; r++) keccak_round<MAD_MASK>(a, KECCAK_RC[r]);
  } else {
#pragma unroll UNROLL
    for (int r = 0; r < 24; r++) keccak_round<MAD_MASK>(a, KECCAK_RC[r]);
  }
}
__device__ __forceinline__ void keccak_f1600(uint64_t (&a)[25]) { keccak_f1600_t<PPD_KECCAK_UNROLL, PPD_KECCAK_MAD_MASK>(a); }

// ---------------------------------------------------------------------------------------------
// Block staging for a byte stream that a thread produces piecewise (RLP headers, child refs,
// values).  Pull model: a thread appends whole units (each <= 136 bytes) to its stage until at
// least one 136-byte rate block is complete, then the WHOLE warp runs the one keccak_f1600 site
// convergently (callers loop warp-uniformly, see ppd_kernels.cu).
//
// The stage is a ring of 2 x 34 32-bit words per thread in shared memory, word-interleaved (word w
// of thread t at stage[w * BLOCK + t]): the bank depends on t only, so every access pattern of a
// warp is conflict-free no matter how far each lane has advanced.  A rate block is exactly one half
// of the ring, so the bytes that overflow a block already sit where the next block starts:
// consuming a block moves no data.
//
// Appending a word costs one funnel shift, one store and the ring-pointer update: the bytes that do
// not yet fill a word are kept in the TOP `sh` bits of `carry`, so the word to store is
// funnelshift_l(carry, x, sh) and the new carry is x itself.  All addresses are 32-bit shared-window
// addresses (explicit ld/st.shared), never generic pointers.
// ---------------------------------------------------------------------------------------------
#define PPD_STAGE_WORDS 68

__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
template <int OFF>
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF) : "memory");
  return v;
}

template <int BLOCK>
struct Stage {
  static constexpr uint32_t STRIDE = 4u * BLOCK;                 // bytes between consecutive words of one thread
  static constexpr uint32_t HALF = 34u * STRIDE, RING = 68u * STRIDE;
  uint32_t lo;     // shared address of this thread's word 0
  uint32_t addr;   // shared address of the next word slot
  uint32_t blk;    // shared address of word 0 of the current block: lo or lo + HALF
  uint32_t carry;  // pending bytes of the word being assembled, in the top `sh` bits
  uint32_t sh;     // 0, 8, 16, 24

  __device__ __forceinline__ void init(uint32_t* smem) {
    lo = (uint32_t)__cvta_generic_to_shared(smem) + 4u * threadIdx.x;
    addr = lo;
    blk = lo;
    carry = 0;
    sh = 0;
  }
  // complete words staged since the start of the current block
  __device__ __forceinline__ uint32_t words() const {
    uint32_t d = addr - blk;
    if ((int32_t)d < 0) d += RING;
    return d / STRIDE;
  }
  __device__ __forceinline__ uint32_t bytes() const { return 4 * words() + (sh >> 3); }
  __device__ __forceinline__ void push_word(uint32_t x) {
    sts32(addr, x);
    addr += STRIDE;
    if (addr == lo + RING) addr = lo;
  }
  __device__ __forceinline__ void put_word(uint32_t x) {
    push_word(__funnelshift_l(carry, x, sh));
    carry = x;
  }
  __device__ __forceinline__ void put_byte(uint32_t b) {
    carry = __funnelshift_r(carry, b, 8);
    sh += 8;
    if (sh == 32) {
      push_word(carry);
      sh = 0;
    }
  }
  // append the low n bytes of x (n = 0..4)
  __device__ __forceinline__ void put_partial(uint32_t x, uint32_t n) {
    if (n == 0) return;
    uint32_t nsh = sh + 8 * n;
    if (nsh >= 32) {
      push_word(__funnelshift_l(carry, x, sh));
      nsh -= 32;
    }
    carry = __funnelshift_rc(carry, x, 8 * n);
    sh = nsh;
  }
  // the pending bytes, low-aligned
  __device__ __forceinline__ uint32_t pending() const { return sh ? carry >> (32 - sh) : 0u; }
  // Keccak padding 0x01 .. 0x80 (original Keccak, as tiny-keccak's Keccak::v256).  Needs bytes() < 136.
  __device__ __forceinline__ void pad() {
    const uint32_t last = blk + 33u * STRIDE;
    uint32_t v = pending() | (0x01u << sh);
    uint32_t p = addr;  // words() < 34: the slot of the partial word, inside the current half
    while (p != last) {
      sts32(p, v);
      v = 0;
      p += STRIDE;
    }
    sts32(last, v | 0x80000000u);
  }
  // after a block was absorbed: the overflow words are already at the start of the other half
  __device__ __forceinline__ void consume_block() { blk = (blk == lo) ? lo + HALF : lo; }
  // word K of the current block; flush_partial() first if the last word may be incomplete
  template <int K>
  __device__ __forceinline__ uint32_t word() const {
    return lds32<K * (int)STRIDE>(blk);
  }
  // make the partial word visible in shared memory (for the inline < 32-byte case)
  __device__ __forceinline__ void flush_partial() {
    if (sh) sts32(addr, pending());
  }
};

// ---------------------------------------------------------------------------------------------
// Gather slot: source bytes of a thread's NEXT unit, copied from global memory by cp.async while
// the permutation of the current block runs, so that the fill after it reads shared memory instead
// of waiting on L2.  CHUNKS 16-byte chunks per thread, chunk-interleaved (chunk c of thread t at
// slot[c * BLOCK + t]): 16-byte accesses of a warp are conflict-free, and cp.async needs 16
// contiguous bytes.  Every thread reads only its own chunks, so no barrier is involved:
// cp.async.wait_group 0 makes the copies visible to the thread that issued them.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ uint32_t lds32_at(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

template <int BLOCK, int CHUNKS>
struct Gather {
  static constexpr uint32_t STRIDE = 16u * BLOCK;  // bytes between consecutive chunks of one thread
  static constexpr uint32_t BYTES = 16u * CHUNKS * BLOCK;
  uint32_t lo;  // shared address of this thread's chunk 0

  __device__ __forceinline__ void init(const void* base) { lo = (uint32_t)__cvta_generic_to_shared(base) + 16u * threadIdx.x; }
  __device__ __forceinline__ uint32_t chunk(uint32_t c) const { return lo + c * STRIDE; }
  // 32-bit word i of the slot (word i & 3 of chunk i >> 2)
  __device__ __forceinline__ uint32_t word(uint32_t i) const { return lds32_at(lo + (i >> 2) * STRIDE + 4u * (i & 3)); }
  __device__ __forceinline__ void put_word(uint32_t i, uint32_t v) const { sts32(lo + (i >> 2) * STRIDE + 4u * (i & 3), v); }
};

template <int BLOCK>
__device__ __forceinline__ void absorb_stage(uint64_t (&a)[25], const Stage<BLOCK>& s) {
#define PPD_ABSORB(i) a[i] ^= ((uint64_t)s.template word<2 * (i) + 1>() << 32) | s.template word<2 * (i)>();
  PPD_ABSORB(0) PPD_ABSORB(1) PPD_ABSORB(2) PPD_ABSORB(3) PPD_ABSORB(4) PPD_ABSORB(5) PPD_ABSORB(6) PPD_ABSORB(7) PPD_ABSORB(8)
  PPD_ABSORB(9) PPD_ABSORB(10) PPD_ABSORB(11) PPD_ABSORB(12) PPD_ABSORB(13) PPD_ABSORB(14) PPD_ABSORB(15) PPD_ABSORB(16)
#undef PPD_ABSORB
}

}  // namespace ppd
