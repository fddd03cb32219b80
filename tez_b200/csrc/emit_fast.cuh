// emit_fast.cuh -- gather + IFile emit for fixed-width records whose stride is a multiple of 16 bytes
// (BASELINE config 2/4: 16 B key + 64 B value).  "Source oriented": every lane moves one aligned 128-bit piece of a
// source record into the shared-memory image of the output bytes (funnel-shifted to its unaligned destination), the
// CTA folds the image into the segment CRC32 (two-level interleaved table CRC, constant per-lane alignment
// multipliers) and streams it to HBM with coalesced 128-bit stores.  CTAs are persistent (grid-stride over tiles) so
// the CRC tables are staged into shared memory once.
#pragma once
#include "sorter_kernels.cuh"

#ifndef TEZGPU_EMIT_MIN_CTAS
#define TEZGPU_EMIT_MIN_CTAS 4
#endif

namespace tezgpu {

constexpr int FE_THREADS = 256;
constexpr int FE_MAX_RECS = 256;
constexpr int FE_IMG_BYTES = 22016;  // 256 records * 82 B + lead + header + EOF, multiple of 16

// the source-oriented kernels build a whole tile in one FE_IMG_BYTES image: at least one record plus the worst-case
// lead (15), segment header (4) and EOF markers (2) must fit.  Larger records take the general kernel (k_emit<true>),
// which splits a tile over several images.
static inline bool fast_emit_fits(uint32_t rec_size) { return (uint64_t)rec_size + 15 + 4 + 2 <= (uint64_t)FE_IMG_BYTES; }

struct TileDesc {
  uint32_t p;      // partition
  uint32_t r0;     // first sorted position
  uint32_t nr;     // records
  uint32_t flags;  // 1 = first tile of the segment, 2 = last tile
  uint64_t abs0;   // file offset of the tile's first byte
  uint64_t after;  // body bytes of the segment that follow this tile's bytes
};

// one entry per emit tile: raw (unconditioned) CRC remainder of the tile's body bytes
struct TileCrc {
  uint32_t raw;
  uint32_t p;
  uint64_t after;
};

__global__ void k_build_tiles(EmitParams e, TileDesc *__restrict__ tiles) {
  uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x;
  if (tile >= e.tile_start[e.P]) return;
  int lo = 0, hi = e.P;  // last p with tile_start[p] <= tile
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (e.tile_start[mid] <= tile) lo = mid; else hi = mid;
  }
  const uint32_t p = (uint32_t)lo;
  const uint32_t ps = e.part_start[p], pe = e.part_start[p + 1];
  const uint32_t k = tile - e.tile_start[p];
  TileDesc d;
  d.p = p;
  d.r0 = ps + k * e.recs_per_tile;
  d.nr = min(e.recs_per_tile, pe - d.r0);
  const bool first = (k == 0), last = (d.r0 + d.nr == pe);
  d.flags = (first ? 1u : 0u) | (last ? 2u : 0u);
  const uint64_t seg0 = e.seg_start[p];
  d.abs0 = seg0 + (first ? 0 : 4 + (uint64_t)(d.r0 - ps) * e.rec_size);
  const uint64_t tile_end = seg0 + 4 + (uint64_t)(d.r0 - ps + d.nr) * e.rec_size + (last ? 2 : 0);
  d.after = (e.seg_start[p + 1] - 4) - tile_end;
  tiles[tile] = d;
}

// folds the per-tile remainders into the per-segment remainder: crc(A||B) = crc(A) * x^(8 len B) xor crc(B)
__global__ void k_crc_combine(const TileCrc *__restrict__ tc, uint32_t ntiles, const CrcTables *__restrict__ t,
                              uint32_t *__restrict__ seg_crc) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  uint32_t p = 0xFFFFFFFFu, val = 0;
  if (i < ntiles) {
    TileCrc c = tc[i];
    p = c.p;
    val = c.raw ? crc_shift_bytes(t, c.raw, c.after) : 0u;
  }
  // tiles are ordered by segment: xor-reduce the runs of equal p inside the warp, one atomic per run
  // (same-address atomics serialise at ~20 ns each)
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t v2 = __shfl_up_sync(0xffffffffu, val, o), p2 = __shfl_up_sync(0xffffffffu, p, o);
    if (lane >= o && p2 == p) val ^= v2;
  }
  uint32_t pn = __shfl_down_sync(0xffffffffu, p, 1);
  if (p != 0xFFFFFFFFu && (lane == 31 || pn != p) && val) atomicXor(&seg_crc[p], val);
}

__device__ __forceinline__ void sts_b8(uint32_t a, uint32_t v) { asm volatile("st.shared.b8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_b16(uint32_t a, uint32_t v) { asm volatile("st.shared.b16 [%0], %1;" ::"r"(a), "h"((unsigned short)v) : "memory"); }
__device__ __forceinline__ void sts_b32(uint32_t a, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_v4(uint32_t a, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// stores 16 bytes at an arbitrary shared-memory byte address without touching neighbouring bytes
__device__ __forceinline__ void sts16_unaligned(uint32_t a, uint4 v) {
  const uint32_t al = a & 3u;
  if (al == 0) {
    if ((a & 15u) == 0) sts_v4(a, v);
    else { sts_b32(a, v.x); sts_b32(a + 4, v.y); sts_b32(a + 8, v.z); sts_b32(a + 12, v.w); }
  } else if (al == 2) {
    sts_b16(a, v.x & 0xFFFFu);
    sts_b32(a + 2, __funnelshift_r(v.x, v.y, 16));
    sts_b32(a + 6, __funnelshift_r(v.y, v.z, 16));
    sts_b32(a + 10, __funnelshift_r(v.z, v.w, 16));
    sts_b16(a + 14, v.w >> 16);
  } else if (al == 1) {
    sts_b8(a, v.x & 0xFFu);
    sts_b16(a + 1, (v.x >> 8) & 0xFFFFu);
    sts_b32(a + 3, __funnelshift_r(v.x, v.y, 24));
    sts_b32(a + 7, __funnelshift_r(v.y, v.z, 24));
    sts_b32(a + 11, __funnelshift_r(v.z, v.w, 24));
    sts_b8(a + 15, v.w >> 24);
  } else {
    sts_b8(a, v.x & 0xFFu);
    sts_b32(a + 1, __funnelshift_r(v.x, v.y, 8));
    sts_b32(a + 5, __funnelshift_r(v.y, v.z, 8));
    sts_b32(a + 9, __funnelshift_r(v.z, v.w, 8));
    sts_b16(a + 13, (v.w >> 8) & 0xFFFFu);
    sts_b8(a + 15, v.w >> 24);
  }
}

__device__ __forceinline__ uint4 ldg_stream_v4(const void *p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream_v4(void *p, uint4 v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

struct FastEmitParams {
  EmitParams e;
  const TileDesc *tiles;
  TileCrc *tile_crc;
  uint32_t ntiles;
  uint32_t cpr;        // 16-byte pieces per source record (stride / 16)
  uint32_t cpr_magic;  // floor(2^32 / cpr) + 1
  uint32_t stride;
};

// byte offset in kv of record ri's key: explicit array, arithmetic over the run table, or packed
__device__ __forceinline__ uint64_t fast_source_offset(const Records &rec, uint32_t ri, uint32_t stride, uint32_t p) {
  if (rec.use_runs) return run_record_off_p(rec.runs, p, ri) + rec.runs.hdr_len;   // p: the tile's partition
  return rec.key_off ? rec.key_off[ri] : (uint64_t)ri * stride;
}

#ifndef TEZGPU_CRC_SHFL
#define TEZGPU_CRC_SHFL 1
#endif

template <int UNROLL, bool ALIGNED>
__global__ void __launch_bounds__(FE_THREADS, TEZGPU_EMIT_MIN_CTAS) k_emit_fast(FastEmitParams fp) {
  __shared__ __align__(16) uint8_t s_img[FE_IMG_BYTES];
  __shared__ uint32_t s_idx[2][FE_MAX_RECS];                    // record indices of the current / next tile
  __shared__ uint64_t s_off[ALIGNED ? 1 : 2][ALIGNED ? 1 : FE_MAX_RECS];  // source offsets (explicit-offset mode)
  __shared__ uint32_t s_tab[4 * 256];    // slice-by-4 tables
  __shared__ uint32_t s_adv[4 * 256];    // * x^(32*(4*FE_THREADS-3)): skip to this thread's next 16-byte chunk
  __shared__ uint32_t s_adv32[4 * 256];  // * x^(32*128): second-level fold
  __shared__ uint32_t s_part[FE_THREADS];

  const EmitParams &e = fp.e;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < 4 * 256; i += FE_THREADS) {
    s_tab[i] = (&e.crc->slice[0][0])[i];
    s_adv[i] = (&e.crc->advc[0][0])[i];
    s_adv32[i] = (&e.crc->adv128[0][0])[i];
  }
  // constant alignment multipliers: x^(32*(31-lane)) for the final in-warp fold
  const uint32_t lane_pow = e.crc->pow_word[4 * (31 - lane)];
#if TEZGPU_CRC_SHFL
  // the two maps of the chunk-interleaved checksum as warp-resident 5-bit digit tables (crc32.cuh): "next word"
  // (* x^32) and "skip to this thread's next chunk" (* x^(32*(4*FE_THREADS-3))), built from the global byte tables
  WarpLinearMap m_word, m_skip;
  {
    const uint32_t *gt = &e.crc->slice[0][0], *ga = &e.crc->advc[0][0];
    m_word.init([&](uint32_t x) { return gt[768 + (x & 0xFF)] ^ gt[512 + ((x >> 8) & 0xFF)] ^ gt[256 + ((x >> 16) & 0xFF)] ^ gt[x >> 24]; }, lane);
    m_skip.init([&](uint32_t x) { return ga[x & 0xFF] ^ ga[256 + ((x >> 8) & 0xFF)] ^ ga[512 + ((x >> 16) & 0xFF)] ^ ga[768 + (x >> 24)]; }, lane);
  }
#endif
  const uint32_t img_base = (uint32_t)__cvta_generic_to_shared(s_img);
  const uint8_t *__restrict__ kv = e.rec.kv;
  const uint8_t *kv_end = kv + e.rec.kv_bytes;
  const uint32_t rec_size = e.rec_size, hdr_len = e.fixed_hdr_len, stride = fp.stride;

  // software pipeline over the tiles of this CTA: the descriptor and the record indices (and source offsets) of the
  // NEXT tile are fetched while the current one is gathered / checksummed, so their DRAM latency is off the critical path
  TileDesc td_next;
  if (blockIdx.x < fp.ntiles) {
    td_next = fp.tiles[blockIdx.x];
    if ((uint32_t)tid < td_next.nr) {
      const uint32_t ri = e.order[td_next.r0 + tid];
      s_idx[0][tid] = ri;
      if (!ALIGNED) s_off[0][tid] = fast_source_offset(e.rec, ri, stride, td_next.p);
    }
  }
  uint32_t buf = 0;
  for (uint32_t tile = blockIdx.x; tile < fp.ntiles; tile += gridDim.x, buf ^= 1u) {
    const TileDesc td = td_next;
    const uint32_t nr = td.nr;
    const bool first_tile = td.flags & 1u, last_tile = td.flags & 2u;
    const uint32_t tile_n = tile + gridDim.x;
    if (tile_n < fp.ntiles) td_next = fp.tiles[tile_n];  // consumed after the gather below
    __syncthreads();  // previous tile fully written out; tables / first indices loaded
    const uint32_t *__restrict__ c_idx = s_idx[buf];
    const uint64_t *__restrict__ c_off = s_off[ALIGNED ? 0 : buf];
    const uint64_t abs0 = td.abs0;
    const uint32_t lead = (uint32_t)(abs0 & 15u);
    const uint32_t rec0 = lead + (first_tile ? 4u : 0u);            // image offset of the first record
    const uint32_t body_end = rec0 + nr * rec_size + (last_tile ? 2u : 0u);  // image end

    // ---- gather: lane <-> (record j, 16-byte piece c); all loads of a thread are issued before its stores
    const uint32_t npieces = nr * fp.cpr;
    const uint32_t half_up = (nr + 1) >> 1;
    for (uint32_t q0 = tid; q0 < npieces; q0 += FE_THREADS * UNROLL) {
      uint4 v[UNROLL];
      uint32_t dst[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; u++) {
        uint32_t q = q0 + u * FE_THREADS;
        if (q < npieces) {
          uint32_t jp = fp.cpr == 1 ? q : __umulhi(q, fp.cpr_magic);
          uint32_t c = q - jp * fp.cpr;
          // even records first, then odd ones: the destination alignment (mod 4) alternates with the record parity
          // when the emitted record size is 2 mod 4, so this keeps a warp on one store path
          uint32_t j = jp < half_up ? 2u * jp : 2u * (jp - half_up) + 1u;
          if (ALIGNED) {
            v[u] = ldg_stream_v4(kv + (uint64_t)c_idx[j] * stride + 16u * c);
          } else {
            // records at arbitrary byte offsets (parsed IFile segments): two aligned 128-bit loads + funnel shift;
            // the neighbouring lane's loads hit the same lines in L1
            const uint8_t *a = kv + c_off[j] + 16u * c;
            const uint32_t sh = (uint32_t)((uintptr_t)a & 15u);
            const uint4 *pa = reinterpret_cast<const uint4 *>(a - sh);
            uint4 lo4 = load16_clamped(reinterpret_cast<const uint8_t *>(pa), kv, kv_end);
            uint4 hi4 = sh ? load16_clamped(reinterpret_cast<const uint8_t *>(pa + 1), kv, kv_end) : lo4;
            const uint32_t bsh = (sh & 3u) * 8u;
            uint32_t w0, w1, w2, w3, w4;
            switch (sh >> 2) {
              case 0: w0 = lo4.x; w1 = lo4.y; w2 = lo4.z; w3 = lo4.w; w4 = hi4.x; break;
              case 1: w0 = lo4.y; w1 = lo4.z; w2 = lo4.w; w3 = hi4.x; w4 = hi4.y; break;
              case 2: w0 = lo4.z; w1 = lo4.w; w2 = hi4.x; w3 = hi4.y; w4 = hi4.z; break;
              default: w0 = lo4.w; w1 = hi4.x; w2 = hi4.y; w3 = hi4.z; w4 = hi4.w; break;
            }
            v[u] = make_uint4(__funnelshift_r(w0, w1, bsh), __funnelshift_r(w1, w2, bsh), __funnelshift_r(w2, w3, bsh),
                              __funnelshift_r(w3, w4, bsh));
          }
          dst[u] = img_base + rec0 + j * rec_size + hdr_len + 16u * c;
        }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; u++) {
        uint32_t q = q0 + u * FE_THREADS;
        if (q < npieces) sts16_unaligned(dst[u], v[u]);
      }
    }
    // ---- next tile's record indices (latency hidden behind the framing / checksum / write-out of this tile)
    if (tile_n < fp.ntiles && (uint32_t)tid < td_next.nr) {
      const uint32_t ri = e.order[td_next.r0 + tid];
      s_idx[buf ^ 1u][tid] = ri;
      if (!ALIGNED) s_off[buf ^ 1u][tid] = fast_source_offset(e.rec, ri, stride, td_next.p);
    }
    // ---- framing: vint(klen) vint(vlen) in front of every record, segment header, EOF markers
    if ((uint32_t)tid < nr) {
      uint32_t a = img_base + rec0 + tid * rec_size;
      for (uint32_t b = 0; b < hdr_len; b++) sts_b8(a + b, e.fixed_hdr[b]);
    }
    if (tid == 0) {
      if (first_tile) { s_img[lead] = 'T'; s_img[lead + 1] = 'I'; s_img[lead + 2] = 'F'; s_img[lead + 3] = 0; }
      if (last_tile) { s_img[body_end - 2] = 0xFF; s_img[body_end - 1] = 0xFF; }
    }
    __syncthreads();

    // ---- fused CRC + write-out.  Every thread streams its 16-byte chunks of the image to HBM and folds the same
    // registers into the checksum: thread t owns the chunks whose distance from the end of the body is == T-1-t
    // (mod T), so its partial always needs the constant alignment multiplier x^(128*(T-1-t)).  Leading bytes of the
    // first chunk that precede the body are masked to zero (no effect on a remainder with zero initial value); the
    // trailing partial chunk is folded bytewise by lane 0.
    const uint32_t cb0 = rec0, cb1 = body_end;
    const uint32_t ca = cb0 >> 4, cz = cb1 >> 4;  // whole chunks [ca, cz) belong to the body (first one masked)
    {
      uint8_t *dstg = e.out + (abs0 - lead);
      uint32_t c = 0;
      if (cz > ca) {
        const uint32_t Cn = cz - ca;
#if TEZGPU_CRC_SHFL
        // uniform trip count for the whole CTA (the maps are warp collectives); a thread whose chunk index is still
        // negative folds zeros, which stay zero
        const uint32_t iters = (Cn + FE_THREADS - 1) / FE_THREADS;
        const int32_t last_i = (int32_t)Cn - FE_THREADS + tid;
        int32_t i = last_i - (int32_t)(iters - 1) * FE_THREADS;
        for (uint32_t it = 0; it < iters; it++, i += FE_THREADS) {
          uint4 v = make_uint4(0, 0, 0, 0);
          if (i >= 0) {
            const uint32_t b0 = 16u * (ca + (uint32_t)i);
            v = *reinterpret_cast<const uint4 *>(s_img + b0);
            if (b0 >= lead) stg_stream_v4(dstg + b0, v);
            else for (uint32_t x = lead; x < b0 + 16u; x++) dstg[x] = s_img[x];  // ragged first chunk of the tile
            if (i == 0 && (cb0 & 15u)) {  // zero the bytes before the body (segment header / previous tile's bytes)
              const uint32_t skip = cb0 & 15u;
              uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
              for (uint32_t k = 0; k < 4; k++) {
                if (skip >= 4 * k + 4) w[k] = 0;
                else if (skip > 4 * k) w[k] &= 0xFFFFFFFFu << (8u * (skip - 4 * k));
              }
              v = make_uint4(w[0], w[1], w[2], w[3]);
            }
          }
          uint32_t x = m_word.apply(c ^ v.x) ^ v.y;
          x = m_word.apply(x) ^ v.z;
          x = m_word.apply(x) ^ v.w;
          c = (it + 1 == iters) ? m_word.apply(x) : m_skip.apply(x);
        }
#else
        if (Cn + tid >= FE_THREADS) {
          const uint32_t last_i = Cn - FE_THREADS + tid;
          for (uint32_t i = last_i % FE_THREADS; i <= last_i; i += FE_THREADS) {
            const uint32_t b0 = 16u * (ca + i);
            uint4 v = *reinterpret_cast<const uint4 *>(s_img + b0);
            if (b0 >= lead) stg_stream_v4(dstg + b0, v);
            else for (uint32_t x = lead; x < b0 + 16u; x++) dstg[x] = s_img[x];  // ragged first chunk of the tile
            if (i == 0 && (cb0 & 15u)) {  // zero the bytes before the body (segment header / previous tile's bytes)
              const uint32_t skip = cb0 & 15u;
              uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
              for (uint32_t k = 0; k < 4; k++) {
                if (skip >= 4 * k + 4) w[k] = 0;
                else if (skip > 4 * k) w[k] &= 0xFFFFFFFFu << (8u * (skip - 4 * k));
              }
              v = make_uint4(w[0], w[1], w[2], w[3]);
            }
            uint32_t x = c ^ v.x;
            x = s_tab[768 + (x & 0xFF)] ^ s_tab[512 + ((x >> 8) & 0xFF)] ^ s_tab[256 + ((x >> 16) & 0xFF)] ^ s_tab[x >> 24];
            x ^= v.y;
            x = s_tab[768 + (x & 0xFF)] ^ s_tab[512 + ((x >> 8) & 0xFF)] ^ s_tab[256 + ((x >> 16) & 0xFF)] ^ s_tab[x >> 24];
            x ^= v.z;
            x = s_tab[768 + (x & 0xFF)] ^ s_tab[512 + ((x >> 8) & 0xFF)] ^ s_tab[256 + ((x >> 16) & 0xFF)] ^ s_tab[x >> 24];
            x ^= v.w;
            if (i == last_i) c = s_tab[768 + (x & 0xFF)] ^ s_tab[512 + ((x >> 8) & 0xFF)] ^ s_tab[256 + ((x >> 16) & 0xFF)] ^ s_tab[x >> 24];
            else c = s_adv[x & 0xFF] ^ s_adv[256 + ((x >> 8) & 0xFF)] ^ s_adv[512 + ((x >> 16) & 0xFF)] ^ s_adv[768 + (x >> 24)];
          }
        }
#endif
      }
      s_part[tid] = c;
      // chunks outside [ca, cz): the tile's leading header-only chunk (cannot happen: header and body share chunk ca
      // or follow it) and the trailing partial chunk
      if (tid == 0) {
        for (uint32_t x = max(lead, 16u * cz); x < body_end; x++) dstg[x] = s_img[x];
        if (ca > (lead >> 4)) for (uint32_t x = lead; x < 16u * ca; x++) dstg[x] = s_img[x];
      }
    }
    __syncthreads();
    if (warp == 0) {
      // level 2: lane l folds partials l, l+32, ... (Horner with x^(128*32)), level 3: align by x^(128*(31-l)), xor-reduce
      uint32_t q = 0;
#pragma unroll
      for (int k = 0; k < FE_THREADS / 32; k++) {
        q = s_adv32[q & 0xFF] ^ s_adv32[256 + ((q >> 8) & 0xFF)] ^ s_adv32[512 + ((q >> 16) & 0xFF)] ^ s_adv32[768 + (q >> 24)];
        q ^= s_part[lane + 32 * k];
      }
      q = crc_multmodp(q, lane_pow);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) q ^= __shfl_xor_sync(0xffffffffu, q, o);
      if (lane == 0) {
        uint32_t raw = q;
        if (cz <= ca) {  // body shorter than one chunk: bytewise from cb0
          raw = 0;
          for (uint32_t b = cb0; b < cb1; b++) raw = s_tab[(raw ^ s_img[b]) & 0xFF] ^ (raw >> 8);
        } else {
          for (uint32_t b = 16u * cz; b < cb1; b++) raw = s_tab[(raw ^ s_img[b]) & 0xFF] ^ (raw >> 8);
        }
        TileCrc tc;
        tc.raw = raw;
        tc.p = td.p;
        tc.after = td.after;
        fp.tile_crc[tile] = tc;
      }
    }
  }
}


}  // namespace tezgpu
