// emit_pipe.cuh -- software-pipelined variant of the source-oriented emit kernel (emit_fast.cuh) for packed,
// 16-byte aligned fixed-width records.
//
// What the profile of k_emit_fast showed (profiles/r01_emit_shfl_*): no pipe saturated (LSU data pipe 65 %, issue 53 %),
// 25 % of the warp samples waiting on the gather's global loads, 19 % at barriers (11 % of it behind warp 0 folding
// the tile's partial checksums while seven warps idle).  This kernel keeps the same tile algorithm and byte-exact
// output but reorders the work of a persistent CTA:
//   * the 128-bit gather loads of tile N+1 are issued into registers BEFORE the checksum / write-out loop of tile N
//     and stored to the image after it (record indices are fetched two tiles ahead, tile descriptors three), so the
//     DRAM latency of the random gather hides behind ~190 instructions per thread-chunk of CRC work;
//   * the per-tile second-level checksum fold is deferred: partials of FE4_BATCH tiles are parked in shared memory
//     and folded together, one tile per warp, so no warp waits for another's serial fold;
//   * two barriers per tile instead of three.
#pragma once
#include "emit_fast.cuh"

#ifndef TEZGPU_EMIT4_MIN_CTAS
#define TEZGPU_EMIT4_MIN_CTAS 3
#endif
#ifndef TEZGPU_EMIT4_MAP16
#define TEZGPU_EMIT4_MAP16 0
#endif

namespace tezgpu {

constexpr int FE4_BATCH = FE_THREADS / 32;  // one parked tile per warp
constexpr int FE4_UNROLL = TEZGPU_EMIT4_MAP16 ? 6 : 5;  // gather rounds held in registers

// can a tile of `recs` records with `cpr` pieces each be gathered in FE4_UNROLL rounds?  Both maps need cpr <= 8: the
// packed piece map of full tiles (k_emit_fast4) keeps 16c in a 7-bit field, so piece 8 and up would alias piece c % 8.
static inline bool emit4_fits(uint32_t recs, uint32_t cpr) {
#if TEZGPU_EMIT4_MAP16
  const uint32_t rph = 16u / cpr;
  return cpr <= 8 && 16ull * ((recs + rph - 1) / rph) <= (uint64_t)FE4_UNROLL * FE_THREADS;
#else
  return cpr <= 8 && (uint64_t)recs * cpr <= (uint64_t)FE4_UNROLL * FE_THREADS;
#endif
}

struct FoldMeta {
  uint4 tail;       // the 16-byte chunk holding the bytes the chunk loop did not fold
  uint32_t tile;
  uint32_t start;   // byte range [start, end) of `tail` to fold bytewise
  uint32_t end;
  uint32_t tiny;    // 1: the whole body lies inside `tail` (no whole chunk): start from a zero remainder
};

__device__ __forceinline__ uint4 lds_v4(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}

// SUBS = 1: one 256-thread group per CTA, TEZGPU_EMIT4_MIN_CTAS CTAs per SM, both checksum maps as SHFL digit tables.
// SUBS = 3: one CTA per SM hosts three independent 256-thread groups (named barriers) that share a LANE-PRIVATE copy
//           of the four "next word" byte tables (entry e of table k for lane l lives at word (k*256+e)*32+l, always
//           bank l): the look-up that runs three times per chunk becomes 4 conflict-free LDS instead of 7 SHFL.
//           Measured on the SHFL-only kernel: a SHFL occupies the LSU data pipe for two cycles, so its 28 SHFL per
//           chunk cost as much pipe time as the conflicting byte-table look-ups they replaced; the pipe, not issue
//           or DRAM, bounded the kernel.
template <int SUBS>
struct Emit4Smem {
  static constexpr int BATCH = SUBS > 1 ? 4 : FE4_BATCH;
  static constexpr size_t WTAB = SUBS > 1 ? (size_t)4 * 256 * 32 * 4 : 0;
  static constexpr size_t SHARED = WTAB + 256 * 4 + 4 * 256 * 4;
  static constexpr size_t GROUP = FE_IMG_BYTES + 3 * FE_MAX_RECS * 4 + (size_t)BATCH * FE_THREADS * 4 + (size_t)BATCH * sizeof(FoldMeta);
  static constexpr size_t TOTAL = SHARED + SUBS * GROUP;
};

template <int UNROLL, int SUBS>
__global__ void __launch_bounds__(FE_THREADS * SUBS, SUBS > 1 ? 1 : TEZGPU_EMIT4_MIN_CTAS) k_emit_fast4(FastEmitParams fp) {
  using L = Emit4Smem<SUBS>;
  constexpr int BATCH = L::BATCH;
  extern __shared__ __align__(16) uint8_t smem4[];
  uint32_t *s_wtab = reinterpret_cast<uint32_t *>(smem4);              // [4][256][32] lane-private (SUBS > 1)
  uint32_t *s_tab = reinterpret_cast<uint32_t *>(smem4 + L::WTAB);     // classic byte table (trailing bytes)
  uint32_t *s_adv128 = s_tab + 256;                                    // * x^(32*128): second-level fold
  const int sub = threadIdx.x / FE_THREADS, tid = threadIdx.x % FE_THREADS, lane = tid & 31, warp = tid >> 5;
  uint8_t *gbase = smem4 + L::SHARED + (size_t)sub * L::GROUP;
  uint8_t *s_img = gbase;
  uint32_t(*s_idx)[FE_MAX_RECS] = reinterpret_cast<uint32_t(*)[FE_MAX_RECS]>(gbase + FE_IMG_BYTES);  // tiles N, N+1, N+2
  uint32_t(*s_part)[FE_THREADS] = reinterpret_cast<uint32_t(*)[FE_THREADS]>(gbase + FE_IMG_BYTES + 3 * FE_MAX_RECS * 4);
  FoldMeta *s_meta = reinterpret_cast<FoldMeta *>(gbase + FE_IMG_BYTES + 3 * FE_MAX_RECS * 4 + (size_t)BATCH * FE_THREADS * 4);
  auto group_sync = [&]() {
    if (SUBS == 1) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"r"(sub + 1), "r"(FE_THREADS) : "memory");
  };

  const EmitParams &e = fp.e;
  const uint32_t G = gridDim.x * SUBS, ntiles = fp.ntiles;
  uint32_t tile = blockIdx.x * SUBS + sub;
  if (SUBS > 1)
    for (int i = threadIdx.x; i < 4 * 256 * 32; i += FE_THREADS * SUBS) s_wtab[i] = (&e.crc->slice[0][0])[i >> 5];
  for (int i = threadIdx.x; i < 256; i += FE_THREADS * SUBS) s_tab[i] = e.crc->slice[0][i];
  for (int i = threadIdx.x; i < 4 * 256; i += FE_THREADS * SUBS) s_adv128[i] = (&e.crc->adv128[0][0])[i];
  __syncthreads();
  if (tile >= ntiles) return;
  CrcChunkFoldT<false> cf;  // the chunk fold's linear maps as warp-resident digit tables (crc32.cuh)
  cf.init(e.crc, lane);
  const uint32_t lane_pow = SUBS == 1 ? cf.lane_pow : e.crc->pow_word[4 * (31 - lane)];
  const WarpLinearMap &m_word = cf.w, &m_skip = cf.s;
  const uint32_t *wt = s_wtab + lane;  // this lane's bank
  auto next_word = [&](uint32_t x) -> uint32_t {
    if (SUBS == 1) return m_word.apply(x);
    return wt[(768u + (x & 0xFFu)) << 5] ^ wt[(512u + ((x >> 8) & 0xFFu)) << 5] ^ wt[(256u + ((x >> 16) & 0xFFu)) << 5] ^ wt[(x >> 24) << 5];
  };
  const uint32_t img_base = (uint32_t)__cvta_generic_to_shared(s_img);
  const uint8_t *__restrict__ kv = e.rec.kv;
  const uint32_t rec_size = e.rec_size, hdr_len = e.fixed_hdr_len, stride = fp.stride, cpr = fp.cpr;
  const TileDesc *__restrict__ tiles = fp.tiles;

  // piece slot of a tile <-> (record j, 16-byte piece c).
  // MAP16 = 0: consecutive lanes take consecutive pieces, records straddle the 8-lane quarters a 128-bit warp load is
  //            split into, so a quarter touches the lines of up to three records;
  // MAP16 = 1: every half-warp takes 16/cpr whole records (leftover lanes idle): fewer distinct 128-byte lines per
  //            quarter -> fewer L1 wavefronts for the random gather.
  // Even records first, then odd ones (emit_fast.cuh): keeps a warp on one unaligned-store path.
#if TEZGPU_EMIT4_MAP16
  const uint32_t rph = 16u / cpr;                       // records per half-warp
  const uint32_t hl = tid & 15u, rl = hl / cpr, pc = hl - rl * cpr;
  const bool lane_used = rl < rph;
  auto piece = [&](int u, uint32_t nr, uint32_t &j, uint32_t &c) -> bool {
    const uint32_t jp = (((uint32_t)tid >> 4) + 16u * (uint32_t)u) * rph + rl;
    c = pc;
    const uint32_t half_up = (nr + 1) >> 1;
    j = jp < half_up ? 2u * jp : 2u * (jp - half_up) + 1u;
    return lane_used && jp < nr;
  };
#else
  auto piece = [&](int u, uint32_t nr, uint32_t &j, uint32_t &c) -> bool {
    const uint32_t q = tid + u * FE_THREADS;
    const uint32_t jp = cpr == 1 ? q : __umulhi(q, fp.cpr_magic);
    c = q - jp * cpr;
    const uint32_t half_up = (nr + 1) >> 1;
    j = jp < half_up ? 2u * jp : 2u * (jp - half_up) + 1u;
    return q < nr * cpr;
  };
#endif
  // Full tiles (all but the last of a partition) share one piece map: packed once per thread as
  // j | 16c << 8 | (j * rec_size + hdr_len + 16c) << 15 (16c < 128: emit4_fits admits cpr <= 8 only), so a piece
  // costs an index look-up and one multiply-add instead of the divide / permute arithmetic (which was ~25 % of the
  // kernel's instructions).
  const uint32_t full_nr = e.recs_per_tile;
  uint32_t pk[UNROLL], onmask = 0;
#pragma unroll
  for (int u = 0; u < UNROLL; u++) {
    uint32_t j, c;
    const bool on = piece(u, full_nr, j, c);
    pk[u] = on ? (j | (16u * c) << 8 | (j * rec_size + hdr_len + 16u * c) << 15) : 0u;
    onmask |= on ? 1u << u : 0u;
  }
  uint4 v[UNROLL];
  // all addresses first, then the loads back to back (keeps ptxas from reusing the destination registers of later
  // rounds as temporaries between the loads)
  auto issue_gather = [&](uint32_t nr, const uint32_t *idx) {
    const uint8_t *src[UNROLL];
    bool on[UNROLL];
    if (nr == full_nr) {
#pragma unroll
      for (int u = 0; u < UNROLL; u++) {
        on[u] = (onmask >> u) & 1u;
        src[u] = kv + (uint64_t)idx[pk[u] & 0xFFu] * stride + ((pk[u] >> 8) & 0x7Fu);
      }
    } else {
#pragma unroll
      for (int u = 0; u < UNROLL; u++) {
        uint32_t j, c;
        on[u] = piece(u, nr, j, c);
        src[u] = kv + (uint64_t)idx[on[u] ? j : 0u] * stride + 16u * c;
      }
    }
    if (UNROLL == 5) asm volatile("" : "+l"(src[0]), "+l"(src[1]), "+l"(src[2]), "+l"(src[3]), "+l"(src[UNROLL - 1]));
#pragma unroll
    for (int u = 0; u < UNROLL; u++)
      if (on[u]) v[u] = ldg_stream_v4(src[u]);
  };
  // vint(klen) vint(vlen) of the fixed framing as one 16-bit store when it is two bytes at an even address
  const uint32_t hdr16 = (uint32_t)e.fixed_hdr[0] | (uint32_t)e.fixed_hdr[1] << 8;

  // ---- prologue: descriptors of tiles 0..2 of this CTA, indices of tiles 0 and 1, gather of tile 0 in flight
  uint32_t nr0, fl0, nr1 = 0, fl1 = 0, r0_2 = 0, nr2 = 0;
  uint64_t abs0, abs1 = 0;
  {
    const TileDesc t0 = tiles[tile];
    nr0 = t0.nr; fl0 = t0.flags; abs0 = t0.abs0;
    if ((uint32_t)tid < nr0) s_idx[0][tid] = e.order[t0.r0 + tid];
    if (tile + G < ntiles) {
      const TileDesc t1 = tiles[tile + G];
      nr1 = t1.nr; fl1 = t1.flags; abs1 = t1.abs0;
      if ((uint32_t)tid < nr1) s_idx[1][tid] = e.order[t1.r0 + tid];
    }
    if (tile + 2 * (uint64_t)G < ntiles) { r0_2 = tiles[tile + 2 * G].r0; nr2 = tiles[tile + 2 * G].nr; }
  }
  group_sync();
  issue_gather(nr0, s_idx[0]);

  uint32_t n_it = 0, slot = 0;
  for (;; tile += G, n_it++) {
    const bool has1 = tile + G < ntiles, has2 = tile + 2 * (uint64_t)G < ntiles, has3 = tile + 3 * (uint64_t)G < ntiles;
    const uint32_t nr = nr0;
    const bool first_tile = fl0 & 1u, last_tile = fl0 & 2u;
    const uint32_t lead = (uint32_t)(abs0 & 15u);
    const uint32_t rec0 = lead + (first_tile ? 4u : 0u);
    const uint32_t body_end = rec0 + nr * rec_size + (last_tile ? 2u : 0u);

    // ---- prefetches that are consumed at the end of this iteration / in the next one
    uint32_t r_idx = 0, r0_3 = 0, nr3 = 0, nr2n = 0, fl2n = 0;
    uint64_t abs2n = 0;
    if (has2) {
      if ((uint32_t)tid < nr2) r_idx = e.order[r0_2 + tid];
      const TileDesc *t2 = tiles + tile + 2 * (uint64_t)G;
      nr2n = t2->nr; fl2n = t2->flags; abs2n = t2->abs0;
    }
    if (has3) { const TileDesc *t3 = tiles + tile + 3 * (uint64_t)G; r0_3 = t3->r0; nr3 = t3->nr; }

    // ---- this tile's pieces (loaded during the previous iteration) -> image; framing
    if (nr == full_nr) {
#pragma unroll
      for (int u = 0; u < UNROLL; u++)
        if ((onmask >> u) & 1u) sts16_unaligned(img_base + rec0 + (pk[u] >> 15), v[u]);
    } else {
#pragma unroll
      for (int u = 0; u < UNROLL; u++) {
        uint32_t j, c;
        if (piece(u, nr, j, c)) sts16_unaligned(img_base + rec0 + j * rec_size + hdr_len + 16u * c, v[u]);
      }
    }
    if ((uint32_t)tid < nr) {
      const uint32_t a = img_base + rec0 + tid * rec_size;
      if (hdr_len == 2 && !(a & 1u)) sts_b16(a, hdr16);
      else for (uint32_t b = 0; b < hdr_len; b++) sts_b8(a + b, e.fixed_hdr[b]);
    }
    if (tid == 0) {
      if (first_tile) { s_img[lead] = 'T'; s_img[lead + 1] = 'I'; s_img[lead + 2] = 'F'; s_img[lead + 3] = 0; }
      if (last_tile) { s_img[body_end - 2] = 0xFF; s_img[body_end - 1] = 0xFF; }
    }
    group_sync();  // (B) image complete

    // ---- gather of the next tile goes out now; it lands while this tile is checksummed and written
    if (has1) issue_gather(nr1, s_idx[(n_it + 1) % 3]);

    // ---- fused CRC + write-out (emit_fast.cuh): thread t owns the chunks at distance == T-1-t (mod T) from the end
    const uint32_t cb0 = rec0, cb1 = body_end;
    const uint32_t ca = cb0 >> 4, cz = cb1 >> 4;
    uint8_t *dstg = e.out + (abs0 - lead);
    uint32_t c = 0;
    if (cz > ca) {
      const uint32_t Cn = cz - ca;
      const uint32_t iters = (Cn + FE_THREADS - 1) / FE_THREADS;
      int32_t i = (int32_t)Cn + tid - (int32_t)(iters * FE_THREADS);
      uint32_t sa = img_base + 16u * (uint32_t)((int32_t)ca + i);
      uint8_t *gp = dstg + 16ll * ((int64_t)ca + i);
      for (uint32_t it = 0; it < iters; it++, i += FE_THREADS, sa += 16u * FE_THREADS, gp += 16 * FE_THREADS) {
        if (i + (31 - lane) < 0) continue;  // no lane of this warp owns a chunk yet (first, ragged round only)
        uint4 w = make_uint4(0, 0, 0, 0);
        if (i >= 0) {
          w = lds_v4(sa);
          if (i == 0) {
            const uint32_t b0 = 16u * ca;
            if (b0 >= lead) stg_stream_v4(gp, w);
            else for (uint32_t x = lead; x < b0 + 16u; x++) dstg[x] = s_img[x];  // ragged first chunk of the tile
            const uint32_t skip = cb0 & 15u;  // bytes before the body (segment header / previous tile) fold as zero
            if (skip) {
              uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
              for (uint32_t k = 0; k < 4; k++) {
                if (skip >= 4 * k + 4) ww[k] = 0;
                else if (skip > 4 * k) ww[k] &= 0xFFFFFFFFu << (8u * (skip - 4 * k));
              }
              w = make_uint4(ww[0], ww[1], ww[2], ww[3]);
            }
          } else {
            stg_stream_v4(gp, w);
          }
        }
        if (SUBS == 1) {
          c = cf.fold(c, w, it + 1 == iters);
        } else {
          uint32_t x = next_word(c ^ w.x) ^ w.y;
          x = next_word(x) ^ w.z;
          x = next_word(x) ^ w.w;
          c = (it + 1 == iters) ? next_word(x) : m_skip.apply(x);
        }
      }
    }
    s_part[slot][tid] = c;
    if (tid == 0) {
      // bytes outside the whole chunks: trailing partial chunk, and a leading header-only chunk
      for (uint32_t x = max(lead, 16u * cz); x < body_end; x++) dstg[x] = s_img[x];
      if (ca > (lead >> 4)) for (uint32_t x = lead; x < 16u * ca; x++) dstg[x] = s_img[x];
      FoldMeta m;
      m.tail = *reinterpret_cast<const uint4 *>(s_img + 16u * cz);  // cz == ca when there is no whole chunk
      m.tile = tile;
      m.tiny = cz > ca ? 0u : 1u;
      m.start = cz > ca ? 0u : (cb0 & 15u);
      m.end = cb1 & 15u;
      s_meta[slot] = m;
    }
    if (has2) s_idx[(n_it + 2) % 3][tid] = r_idx;
    slot++;
    group_sync();  // (C) image free, partials / indices visible

    if (slot == (uint32_t)BATCH || !has1) {
      // ---- deferred second level: warp w folds parked tile w.  lane l folds partials l, l+32, ... (Horner with
      // x^(128*32)), aligns by x^(128*(31-l)), xor-reduce; lane 0 appends the trailing bytes
      if ((uint32_t)warp < slot) {
        uint32_t q = 0;
#pragma unroll
        for (int k = 0; k < FE_THREADS / 32; k++) {
          q = s_adv128[q & 0xFF] ^ s_adv128[256 + ((q >> 8) & 0xFF)] ^ s_adv128[512 + ((q >> 16) & 0xFF)] ^ s_adv128[768 + (q >> 24)];
          q ^= s_part[warp][lane + 32 * k];
        }
        q = crc_multmodp(q, lane_pow);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q ^= __shfl_xor_sync(0xffffffffu, q, o);
        if (lane == 0) {
          const FoldMeta m = s_meta[warp];
          const uint32_t tw[4] = {m.tail.x, m.tail.y, m.tail.z, m.tail.w};
          uint32_t raw = m.tiny ? 0u : q;
          for (uint32_t b = m.start; b < m.end; b++) {
            const uint32_t byte = (tw[b >> 2] >> (8u * (b & 3u))) & 0xFFu;
            raw = s_tab[(raw ^ byte) & 0xFF] ^ (raw >> 8);
          }
          const TileDesc td = tiles[m.tile];
          TileCrc tc;
          tc.raw = raw;
          tc.p = td.p;
          tc.after = td.after;
          fp.tile_crc[m.tile] = tc;
        }
      }
      slot = 0;
      // the parked rows are rewritten only after barrier (B) of the next iteration, which every folding warp joins
    }
    if (!has1) break;
    // the descriptor prefetches are consumed HERE: without this the compiler renames them straight into the next
    // iteration, where their scoreboard is shared with the freshly issued gather loads and the first use stalls on
    // those (measured: 20 % of all warp samples on one integer add in the middle of the gather)
    asm volatile("" : "+r"(nr2n), "+r"(fl2n), "+l"(abs2n), "+r"(r0_3), "+r"(nr3));
    nr0 = nr1; fl0 = fl1; abs0 = abs1;
    nr1 = nr2n; fl1 = fl2n; abs1 = abs2n;
    r0_2 = r0_3; nr2 = nr3;
  }
}

}  // namespace tezgpu
