// crc32.cuh -- CRC-32 (poly 0xEDB88320, the IFileOutputStream / PureJavaCrc32 checksum,
// SORT/IFileOutputStream.java:53-90, SORT/TezSpillRecord.java:111-146) for parallel use on the device.
//
// The per-segment checksum of an IFile body is sequential by definition; on the device every emit tile computes the
// standard CRC of its own bytes and folds it into the segment checksum with
//     crc(A || B) = crc(A) * x^(8*len(B))  xor  crc(B)          (GF(2)[x] / P, reflected bit order)
// so tiles combine with one atomicXor each.  Powers of x come from three 4096-entry tables (x^(8*a0),
// x^(8*4096*a1), x^(8*2^24*a2)) computed once on the host.
#pragma once
#include "common.cuh"

namespace tezgpu {

constexpr uint32_t CRC_POLY = 0xEDB88320u;

// a(x) * b(x) mod P, reflected representation (bit 31 = x^0)
__host__ __device__ __forceinline__ uint32_t crc_multmodp(uint32_t a, uint32_t b) {
  uint32_t p = 0;
#ifdef __CUDA_ARCH__
#pragma unroll 4
#endif
  for (int i = 0; i < 32; i++) {
    p ^= b & (0u - ((a >> (31 - i)) & 1u));
    b = (b >> 1) ^ (CRC_POLY & (0u - (b & 1u)));
  }
  return p;
}

struct CrcTables {
  uint32_t slice[4][256];   // slice-by-4 byte tables: slice[k][b] = (b * x^(8*(k+1))) mod P, k = 0 is the classic table
  uint32_t adv[4][256];     // multiply-by-x^(32*EMIT_CRC_STRIDE_WORDS) byte tables (interleaved per-thread streams)
  uint32_t adv32[4][256];   // multiply-by-x^(32*32) byte tables (second-level fold of the per-thread partials)
  uint32_t advc[4][256];    // multiply-by-x^(32*(4*stride-3)): 16-byte-chunk interleave (fused CRC + write-out)
  uint32_t adv128[4][256];  // multiply-by-x^(32*128): second-level fold of chunk-interleaved partials
  uint32_t advc2[4][256];   // multiply-by-x^(32*(4*stride-1)): the "skip" of advc composed with two "next word" steps
  uint32_t einv;            // x^(-128*(stride-1)): undoes the skip the two-deep chunk fold applies after a thread's LAST chunk
  uint32_t pow_word[512];   // x^(32*j), j < 512
  uint32_t pow0[4096];      // x^(8*a)
  uint32_t pow1[4096];      // x^(8*4096*a)
  uint32_t pow2[4096];      // x^(8*2^24*a)
};

static inline uint32_t crc_host_xpow8(uint64_t nbytes) {
  // x^(8*nbytes) mod P by square-and-multiply
  uint32_t result = 0x80000000u;  // x^0
  uint32_t base = 0x00800000u;    // x^8
  while (nbytes) {
    if (nbytes & 1) result = crc_multmodp(result, base);
    base = crc_multmodp(base, base);
    nbytes >>= 1;
  }
  return result;
}

// x^nbits mod P by square-and-multiply
static inline uint32_t crc_host_xpow_bits(uint64_t nbits) {
  uint32_t result = 0x80000000u;  // x^0
  uint32_t base = 0x40000000u;    // x^1
  while (nbits) {
    if (nbits & 1) result = crc_multmodp(result, base);
    base = crc_multmodp(base, base);
    nbits >>= 1;
  }
  return result;
}
// x^(-nbits) mod P: the CRC-32 polynomial is primitive, x has order 2^32 - 1 (checked on the CPU: tests/test_abi_cpu.py)
static inline uint32_t crc_host_xpow_bits_inv(uint64_t nbits) {
  const uint64_t ord = 0xFFFFFFFFull;
  return crc_host_xpow_bits((ord - nbits % ord) % ord);
}

static inline void crc_build_tables(CrcTables &t, int stride_words) {
  for (uint32_t i = 0; i < 256; i++) {
    uint32_t c = i;
    for (int k = 0; k < 8; k++) c = (c & 1) ? CRC_POLY ^ (c >> 1) : (c >> 1);
    t.slice[0][i] = c;
  }
  for (uint32_t i = 0; i < 256; i++)
    for (int k = 1; k < 4; k++) t.slice[k][i] = (t.slice[k - 1][i] >> 8) ^ t.slice[0][t.slice[k - 1][i] & 0xFF];
  // adv[k][b] = (b << 8k) * x^(32*stride_words): a register value v with byte b at bits [8k,8k+8)
  uint32_t xs = crc_host_xpow8((uint64_t)4 * (uint64_t)stride_words);
  for (int k = 0; k < 4; k++)
    for (uint32_t b = 0; b < 256; b++) t.adv[k][b] = crc_multmodp(b << (8 * k), xs);
  uint32_t x32w = crc_host_xpow8((uint64_t)4 * 32);
  for (int k = 0; k < 4; k++)
    for (uint32_t b = 0; b < 256; b++) t.adv32[k][b] = crc_multmodp(b << (8 * k), x32w);
  uint32_t xc = crc_host_xpow8((uint64_t)4 * (uint64_t)(4 * stride_words - 3)), x128 = crc_host_xpow8((uint64_t)4 * 128);
  for (int k = 0; k < 4; k++)
    for (uint32_t b = 0; b < 256; b++) {
      t.advc[k][b] = crc_multmodp(b << (8 * k), xc);
      t.adv128[k][b] = crc_multmodp(b << (8 * k), x128);
    }
  const uint32_t xc2 = crc_host_xpow8((uint64_t)4 * (uint64_t)(4 * stride_words - 1));
  for (int k = 0; k < 4; k++)
    for (uint32_t b = 0; b < 256; b++) t.advc2[k][b] = crc_multmodp(b << (8 * k), xc2);
  t.einv = crc_host_xpow_bits_inv((uint64_t)128 * (uint64_t)(stride_words - 1));
  for (int j = 0; j < 512; j++) t.pow_word[j] = crc_host_xpow8((uint64_t)4 * (uint64_t)j);
  uint32_t s0 = crc_host_xpow8(1), s1 = crc_host_xpow8(4096), s2 = crc_host_xpow8(1ull << 24);
  t.pow0[0] = t.pow1[0] = t.pow2[0] = 0x80000000u;
  for (int a = 1; a < 4096; a++) {
    t.pow0[a] = crc_multmodp(t.pow0[a - 1], s0);
    t.pow1[a] = crc_multmodp(t.pow1[a - 1], s1);
    t.pow2[a] = crc_multmodp(t.pow2[a - 1], s2);
  }
}

// ---------------------------------------------------------------------------------------------- warp-resident maps
// Every step of the interleaved checksum is a GF(2)-linear map of a 32-bit word ("multiply by a fixed power of x"),
// classically four 256-entry table look-ups in shared memory.  Random byte values make those look-ups collide on
// banks (measured: 58 % of the emit kernel's shared-load wavefronts were replays).  The same map split into seven
// 5-bit digits needs only 32-entry tables, and a 32-entry table is exactly one register across the lanes of a warp:
// digit k of x selects lane (x >> 5k) & 31 of register t[k] with one SHFL -- no shared memory, no conflicts.
// All 32 lanes must execute apply() together (lanes with nothing to fold pass 0, which maps to 0).
struct WarpLinearMap {
  uint32_t t[7];
  // f(v) must be the linear map evaluated with any method (byte tables); lane l keeps f(l << 5k)
  template <typename F>
  __device__ __forceinline__ void init(F f, uint32_t lane) {
#pragma unroll
    for (int k = 0; k < 7; k++) t[k] = f(k < 6 ? lane << (5 * k) : (lane & 3u) << 30);
  }
  __device__ __forceinline__ uint32_t apply(uint32_t x) const {
    // shfl.idx reads b[4:0] of the source-lane operand: no masking needed
    uint32_t r0 = __shfl_sync(0xffffffffu, t[0], (int)x);
    uint32_t r1 = __shfl_sync(0xffffffffu, t[1], (int)(x >> 5));
    uint32_t r2 = __shfl_sync(0xffffffffu, t[2], (int)(x >> 10));
    uint32_t r3 = __shfl_sync(0xffffffffu, t[3], (int)(x >> 15));
    uint32_t r4 = __shfl_sync(0xffffffffu, t[4], (int)(x >> 20));
    uint32_t r5 = __shfl_sync(0xffffffffu, t[5], (int)(x >> 25));
    uint32_t r6 = __shfl_sync(0xffffffffu, t[6], (int)(x >> 30));
    return (r0 ^ r1 ^ r2) ^ (r3 ^ r4 ^ r5) ^ r6;
  }
};

// ---------------------------------------------------------------------------------------------- chunk fold
// Per-thread update of the chunk-interleaved checksum for one 16-byte chunk (w0..w3): with W = "* x^32" (next word)
// and S = "* x^(32*(4T-3))" (skip to this thread's next chunk) the textbook update is the dependent chain
//        c' = S( W( W( W(c ^ w0) ^ w1 ) ^ w2 ) ^ w3 )            -- four table maps deep,
// which leaves a warp waiting on its own arithmetic.  Linearity gives the same value two maps deep:
//        u = W(c ^ w0) ^ w1,   v = W(w2) ^ w3,   c' = (S W^2)(u) ^ S(v)
// -- same number of look-ups (28 SHFL), half the latency, the two halves independent.  The thread's LAST chunk ends
// with W instead of S in the textbook form; the two-deep form applies S there too and the constant factor
// x^(128*(T-1)) this adds to every partial is divided out once, in the per-lane alignment multiplier of the final fold
// (CrcTables::einv; the inverse exists because the CRC-32 polynomial is primitive: tests/test_abi_cpu.py).
// The third digit table costs 7 registers: measured on B200, kernels already at their register cap lose more to the
// spills than they gain (k_emit_fast4 with its gather in registers, at 80: 5.44 -> 6.94 ms, k_emit_fast4u 8.5 -> 9.8 ms),
// kernels with headroom gain a little (k_emit_runs 8.98 -> 8.85 ms) or nothing (k_emit_fast4 with its gather in shared
// memory: 4.99 ms either way).  Hence a template flag per kernel.
template <bool ILP>
struct CrcChunkFoldT {
  WarpLinearMap w, s;
  WarpLinearMap sw2;  // ILP only (dead and eliminated otherwise)
  uint32_t lane_pow;  // x^(128*(31-lane)) [* einv]: alignment of lane l's folded partials in the tile's final fold
  __device__ __forceinline__ void init(const CrcTables *__restrict__ t, uint32_t lane) {
    const uint32_t *gt = &t->slice[0][0], *ga = &t->advc[0][0];
    w.init([&](uint32_t x) { return gt[768 + (x & 0xFF)] ^ gt[512 + ((x >> 8) & 0xFF)] ^ gt[256 + ((x >> 16) & 0xFF)] ^ gt[x >> 24]; }, lane);
    s.init([&](uint32_t x) { return ga[x & 0xFF] ^ ga[256 + ((x >> 8) & 0xFF)] ^ ga[512 + ((x >> 16) & 0xFF)] ^ ga[768 + (x >> 24)]; }, lane);
    lane_pow = t->pow_word[4 * (31 - lane)];
    if (ILP) {
      const uint32_t *g2 = &t->advc2[0][0];
      sw2.init([&](uint32_t x) { return g2[x & 0xFF] ^ g2[256 + ((x >> 8) & 0xFF)] ^ g2[512 + ((x >> 16) & 0xFF)] ^ g2[768 + (x >> 24)]; }, lane);
      lane_pow = crc_multmodp(lane_pow, t->einv);
    }
  }
  // all 32 lanes together (lanes without a chunk pass zeros, which stay zero); last = this is the thread's last chunk
  __device__ __forceinline__ uint32_t fold(uint32_t c, uint4 v, bool last) const {
    if (ILP) {
      const uint32_t u = w.apply(c ^ v.x) ^ v.y;
      const uint32_t r = w.apply(v.z) ^ v.w;
      return sw2.apply(u) ^ s.apply(r);
    }
    uint32_t x = w.apply(c ^ v.x) ^ v.y;
    x = w.apply(x) ^ v.z;
    x = w.apply(x) ^ v.w;
    return last ? w.apply(x) : s.apply(x);
  }
};

// crc * x^(8*nbytes) for nbytes < 2^36
__device__ __forceinline__ uint32_t crc_shift_bytes(const CrcTables *__restrict__ t, uint32_t crc, uint64_t nbytes) {
  uint32_t a0 = (uint32_t)(nbytes & 4095), a1 = (uint32_t)((nbytes >> 12) & 4095), a2 = (uint32_t)((nbytes >> 24) & 4095);
  if (a0) crc = crc_multmodp(crc, t->pow0[a0]);
  if (a1) crc = crc_multmodp(crc, t->pow1[a1]);
  if (a2) crc = crc_multmodp(crc, t->pow2[a2]);
  return crc;
}

}  // namespace tezgpu
