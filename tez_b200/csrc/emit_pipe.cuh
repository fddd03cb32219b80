// emit_pipe.cuh -- software-pipelined variant of the source-oriented emit kernel (emit_fast.cuh) for packed,
// 16-byte aligned fixed-width records.
//
// What the profile of k_emit_fast showed (profiles/r01_emit_shfl_*): no pipe saturated (LSU data pipe 65 %, issue 53 %),
// 25 % of the warp samples waiting on the gather's global loads, 19 % at barriers (11 % of it behind warp 0 folding
// the tile's partial checksums while seven warps idle).  This kernel keeps the same tile algorithm and byte-exact
// output but reorders the work of a persistent CTA:
//   * the gather of tiles N+1 .. N+D is in flight while tile N is imaged, checksummed and written.  In k_emit_fast4<.,1>
//     each thread copies its pieces with cp.async (LDGSTS) into a thread-private ring of D stages in shared memory,
//     so the bytes in flight hold no registers; record indices are fetched D+1 tiles ahead, descriptors D+2;
//   * the per-tile second-level checksum fold is deferred: partials of a batch of tiles are parked in shared memory
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
#ifndef TEZGPU_EMIT4_STAGES
#define TEZGPU_EMIT4_STAGES 1  // depth of k_emit_fast4<.,1>'s cp.async ring (profiles/README.md, round 3: 2 and 3 gain nothing)
#endif

namespace tezgpu {

constexpr int FE4_BATCH = FE_THREADS / 32;  // one parked tile per warp
constexpr int FE4_UNROLL = TEZGPU_EMIT4_MAP16 ? 6 : 5;  // gather rounds per tile
constexpr size_t SM_SMEM_BYTES = 228 * 1024;   // shared memory per SM (sm_100) ...
constexpr size_t SM_SMEM_PER_CTA = 1024;       // ... of which the runtime reserves this much per resident CTA

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
//           Its 219 KB of tables leave no room for a cp.async ring, so its pieces wait in registers (STAGES = 0, the
//           loads of tile N+1 in flight during tile N).
// Per group: image | ring [STAGES][UNROLL][FE_THREADS] x 16 B (piece u of thread t at [s][u][t]: conflict-free) |
// descriptors of tiles N .. N+D+2 | parked fold metadata | record indices of tiles N+D, N+D+1 | parked partials.
// BATCH (tiles parked per fold) is a warp's worth where TEZGPU_EMIT4_MIN_CTAS CTAs still fit an SM, half that otherwise.
template <int SUBS>
struct Emit4Smem {
  static constexpr int STAGES = SUBS > 1 ? 0 : TEZGPU_EMIT4_STAGES;
  static constexpr int DEPTH = STAGES > 0 ? STAGES : 1;  // tiles whose gather is in flight
  static constexpr int NIDX = DEPTH + 1, NDESC = DEPTH + 3;
  static constexpr size_t WTAB = SUBS > 1 ? (size_t)4 * 256 * 32 * 4 : 0;
  static constexpr size_t SHARED = WTAB + 256 * 4 + 4 * 256 * 4;
  static constexpr size_t RING = FE_IMG_BYTES;
  static constexpr size_t DESC = RING + (size_t)STAGES * FE4_UNROLL * FE_THREADS * 16;
  static constexpr size_t META = DESC + NDESC * sizeof(TileDesc);
  static constexpr size_t group_bytes(int batch) {
    return META + (size_t)batch * sizeof(FoldMeta) + NIDX * FE_MAX_RECS * 4 + (size_t)batch * FE_THREADS * 4;
  }
  static constexpr int BATCH =
      SUBS > 1 ? 4 : TEZGPU_EMIT4_MIN_CTAS * (SHARED + group_bytes(FE4_BATCH) + SM_SMEM_PER_CTA) <= SM_SMEM_BYTES ? FE4_BATCH : FE4_BATCH / 2;
  static constexpr size_t IDX = META + (size_t)BATCH * sizeof(FoldMeta);
  static constexpr size_t PART = IDX + NIDX * FE_MAX_RECS * 4;
  static constexpr size_t GROUP = group_bytes(BATCH);
  static constexpr size_t TOTAL = SHARED + SUBS * GROUP;
};
static_assert(TEZGPU_EMIT4_MIN_CTAS * (Emit4Smem<1>::TOTAL + SM_SMEM_PER_CTA) <= SM_SMEM_BYTES, "k_emit_fast4 ring does not fit its CTAs/SM");
static_assert(Emit4Smem<3>::TOTAL + SM_SMEM_PER_CTA <= SM_SMEM_BYTES, "k_emit_fast4<.,3> does not fit an SM");

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int UNROLL, int SUBS>
__global__ void __launch_bounds__(FE_THREADS * SUBS, SUBS > 1 ? 1 : TEZGPU_EMIT4_MIN_CTAS) k_emit_fast4(FastEmitParams fp) {
  using L = Emit4Smem<SUBS>;
  static_assert(UNROLL <= FE4_UNROLL, "ring stage sized for FE4_UNROLL pieces per thread");
  constexpr int BATCH = L::BATCH, D = L::DEPTH;
  constexpr bool RING = L::STAGES > 0;
  extern __shared__ __align__(16) uint8_t smem4[];
  uint32_t *s_wtab = reinterpret_cast<uint32_t *>(smem4);              // [4][256][32] lane-private (SUBS > 1)
  uint32_t *s_tab = reinterpret_cast<uint32_t *>(smem4 + L::WTAB);     // classic byte table (trailing bytes)
  uint32_t *s_adv128 = s_tab + 256;                                    // * x^(32*128): second-level fold
  const int sub = threadIdx.x / FE_THREADS, tid = threadIdx.x % FE_THREADS, lane = tid & 31, warp = tid >> 5;
  uint8_t *gbase = smem4 + L::SHARED + (size_t)sub * L::GROUP;
  uint8_t *s_img = gbase;
  TileDesc *s_desc = reinterpret_cast<TileDesc *>(gbase + L::DESC);                                  // ring of NDESC tiles
  FoldMeta *s_meta = reinterpret_cast<FoldMeta *>(gbase + L::META);
  uint32_t(*s_idx)[FE_MAX_RECS] = reinterpret_cast<uint32_t(*)[FE_MAX_RECS]>(gbase + L::IDX);      // ring of NIDX tiles
  uint32_t(*s_part)[FE_THREADS] = reinterpret_cast<uint32_t(*)[FE_THREADS]>(gbase + L::PART);
  // this thread's slot of piece u in ring stage s: + (s * UNROLL + u) * FE_THREADS * 16
  const uint32_t ring_base = (uint32_t)__cvta_generic_to_shared(gbase + L::RING) + 16u * tid;
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
  uint4 v[UNROLL];  // STAGES = 0: the pieces of the tile in flight
  constexpr uint32_t STAGE_STRIDE = (uint32_t)UNROLL * FE_THREADS * 16;
  // all addresses first, then the loads back to back (keeps ptxas from reusing the destination registers of later
  // rounds as temporaries between the loads)
  auto issue_gather = [&](uint32_t nr, const uint32_t *idx, uint32_t stage) {
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
    for (int u = 0; u < UNROLL; u++) {
      if (!on[u]) continue;
      if (RING) cp_async16(stage + u * FE_THREADS * 16, src[u]);
      else v[u] = ldg_stream_v4(src[u]);
    }
  };
  auto landed = [&](int u, uint32_t stage) -> uint4 { return RING ? lds_v4(stage + u * FE_THREADS * 16) : v[u]; };
  // vint(klen) vint(vlen) of the fixed framing as one 16-bit store when it is two bytes at an even address
  const uint32_t hdr16 = (uint32_t)e.fixed_hdr[0] | (uint32_t)e.fixed_hdr[1] << 8;

  // ---- prologue: descriptors of tiles 0 .. D+1 of this group, indices of tiles 0 .. D, gathers of tiles 0 .. D-1
  // in flight (one cp.async group per tile, also for tiles past the end, so that "tile N landed" is always
  // wait_group D-1)
  for (int k = 0; k < D + 2; k++) {
    const uint64_t t = tile + (uint64_t)k * G;
    if (t >= ntiles) break;
    if (k <= D) {
      const uint32_t r0 = tiles[t].r0, nrk = tiles[t].nr;
      if ((uint32_t)tid < nrk) s_idx[k][tid] = e.order[r0 + tid];
    }
    if (tid < 8) reinterpret_cast<uint32_t *>(s_desc + k)[tid] = reinterpret_cast<const uint32_t *>(tiles + t)[tid];
  }
  group_sync();
#pragma unroll
  for (int k = 0; k < D; k++) {
    if (tile + (uint64_t)k * G < ntiles) issue_gather(s_desc[k].nr, s_idx[k], ring_base + k * STAGE_STRIDE);
    if (RING) cp_async_commit();
  }

  uint32_t n_it = 0, slot = 0, stage = ring_base;  // stage: ring stage of tile N (and of tile N+D)
  for (;; tile += G, n_it++) {
    const bool has1 = tile + G < ntiles;
    const bool hasD = tile + (uint64_t)D * G < ntiles, hasD1 = tile + (D + 1ull) * G < ntiles, hasD2 = tile + (D + 2ull) * G < ntiles;
    const TileDesc &cur = s_desc[n_it % L::NDESC];
    const uint32_t nr = cur.nr, fl = cur.flags;
    const uint64_t abs0 = cur.abs0;
    const bool first_tile = fl & 1u, last_tile = fl & 2u;
    const uint32_t lead = (uint32_t)(abs0 & 15u);
    const uint32_t rec0 = lead + (first_tile ? 4u : 0u);
    const uint32_t body_end = rec0 + nr * rec_size + (last_tile ? 2u : 0u);

    // ---- prefetches that are parked in shared memory at the end of this iteration: indices of tile N+D+1,
    // descriptor of tile N+D+2 (one word per thread of the first eight)
    uint32_t r_idx = 0, d_word = 0;
    if (hasD1) {
      const TileDesc &t1 = s_desc[(n_it + D + 1) % L::NDESC];
      if ((uint32_t)tid < t1.nr) r_idx = e.order[t1.r0 + tid];
    }
    if (hasD2 && tid < 8) d_word = reinterpret_cast<const uint32_t *>(tiles + tile + (D + 2ull) * G)[tid];

    // ---- this tile's pieces (in flight since iteration N-D) -> image
    if (RING) cp_async_wait<D - 1>();  // this thread's copies of tile N have landed (and are visible to it)
    if (nr == full_nr) {
#pragma unroll
      for (int u = 0; u < UNROLL; u++)
        if ((onmask >> u) & 1u) sts16_unaligned(img_base + rec0 + (pk[u] >> 15), landed(u, stage));
    } else {
#pragma unroll
      for (int u = 0; u < UNROLL; u++) {
        uint32_t j, c;
        if (piece(u, nr, j, c)) sts16_unaligned(img_base + rec0 + j * rec_size + hdr_len + 16u * c, landed(u, stage));
      }
    }
    // ---- the gather of tile N+D reuses the stage (or registers) just read; it lands while tiles N .. N+D-1 are
    // checksummed and written.  Every value read from the stage has been stored to the image above: the stores
    // wait for the loads' data, and a thread issues in order, so the copies cannot overwrite a slot before its read.
    if (hasD) issue_gather(s_desc[(n_it + D) % L::NDESC].nr, s_idx[(n_it + D) % L::NIDX], stage);
    if (RING) cp_async_commit();
    stage = (n_it + 1) % D == 0 ? ring_base : stage + STAGE_STRIDE;
    // ---- framing
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
    if (hasD1) s_idx[(n_it + D + 1) % L::NIDX][tid] = r_idx;
    if (hasD2 && tid < 8) reinterpret_cast<uint32_t *>(s_desc + (n_it + D + 2) % L::NDESC)[tid] = d_word;
    slot++;
    group_sync();  // (C) image free, partials / indices / descriptor visible

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
  }
}

}  // namespace tezgpu
