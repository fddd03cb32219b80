// combine.cuh -- device combiner for the sum reducers (MRCombiner + IntSumReducer / LongSumReducer), run between the
// sort and the emit: runCombineProcessor -> ValuesIterator grouping -> reducer -> IFile.Writer.append
// (SORT/PipelinedSorter.java:601-609,815-820; RL/common/ValuesIterator.java:177-201; SORT/IFile.java:443-473).
//
// After the tie phase the sorted order (K, order) and the equal-key flags (same[r] = key at r equals key at r-1) are
// final, and equal keys have equal sort words, hence equal partitions: a group never crosses a partition.
//   1. segmented sum over the sorted positions, reduce / scan / apply over SCAN_TILE tiles with a (flag, sum) carry
//      across tiles (groups may span millions of records);
//   2. pack the m groups as new records (key bytes, big-endian sum) in sorted order, which the unchanged emit writes.
// The sum is taken in 64 bits and truncated to the value width: Java's int / long wrap-around.
#pragma once
#include "sorter_kernels.cuh"

namespace tezgpu {

struct CombineParams {
  Records rec;
  const uint32_t *order;
  const uint8_t *same;
  uint32_t n;
  uint32_t vw;  // value width: 4 (IntWritable) or 8 (LongWritable)
};

// big-endian value of sorted position r's record; a value of the wrong width records the smallest such record index
__device__ __forceinline__ uint64_t comb_value(const CombineParams &c, uint32_t i, uint32_t *__restrict__ bad) {
  uint64_t koff;
  uint32_t klen, vlen;
  record_lookup(c.rec, i, koff, klen, vlen);
  if (vlen != c.vw) {
    atomicMin(bad, i);
    return 0;
  }
  const uint8_t *p = c.rec.kv + ((c.rec.val_off && !c.rec.fixed) ? c.rec.val_off[i] : koff + klen);
  uint64_t v = 0;
  for (uint32_t b = 0; b < c.vw; b++) v = (v << 8) | p[b];
  return v;
}

// (flag, sum) segmented-sum operator: `later` absorbs `earlier` unless a group starts inside `later`
__device__ __forceinline__ void seg_absorb(uint32_t &f, uint64_t &s, uint32_t ef, uint64_t es) {
  if (!f) s += es;
  f |= ef;
}

// block-wide segmented scan of one (flag, sum) per thread: exclusive prefix and block total
template <int THREADS>
__device__ __forceinline__ void block_seg_scan(uint32_t f, uint64_t s, uint32_t &xf, uint64_t &xs, uint32_t &tf, uint64_t &ts,
                                               uint32_t *s_f, uint64_t *s_s) {
  constexpr int NW = THREADS / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t pf = __shfl_up_sync(0xffffffffu, f, o);
    const uint64_t ps = __shfl_up_sync(0xffffffffu, s, o);
    if (lane >= o) seg_absorb(f, s, pf, ps);
  }
  if (lane == 31) { s_f[warp] = f; s_s[warp] = s; }
  __syncthreads();
  uint32_t wf = 0, af = 0;
  uint64_t ws = 0, as = 0;
#pragma unroll
  for (int w = 0; w < NW; w++) {
    const uint32_t ef = s_f[w];
    const uint64_t es = s_s[w];
    if (w < warp) { uint32_t tf2 = ef; uint64_t ts2 = es; seg_absorb(tf2, ts2, wf, ws); wf = tf2; ws = ts2; }
    uint32_t tf3 = ef; uint64_t ts3 = es; seg_absorb(tf3, ts3, af, as); af = tf3; as = ts3;
  }
  __syncthreads();
  uint32_t pf = __shfl_up_sync(0xffffffffu, f, 1);
  uint64_t ps = __shfl_up_sync(0xffffffffu, s, 1);
  if (lane == 0) { pf = 0; ps = 0; }
  seg_absorb(pf, ps, wf, ws);
  xf = pf; xs = ps;
  tf = af; ts = as;
}

// ---- 1. reduce: per tile the (flag, sum) aggregate and the number of group heads; values gathered once into vals
__global__ void __launch_bounds__(SCAN_THREADS)
    k_comb_reduce(CombineParams c, uint64_t *__restrict__ vals, uint32_t *__restrict__ agg_f, uint64_t *__restrict__ agg_s,
                  uint64_t *__restrict__ heads, uint32_t *__restrict__ bad) {
  __shared__ uint32_t s_f[SCAN_THREADS / 32];
  __shared__ uint64_t s_s[SCAN_THREADS / 32], s_w[SCAN_THREADS / 32];
  const uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_IPT;  // blocked: a thread owns 8 consecutive
  uint32_t f = 0, h = 0;
  uint64_t s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_IPT; k++) {
    const uint32_t r = base + k;
    if (r < c.n) {
      const uint64_t v = comb_value(c, c.order[r], bad);
      vals[r] = v;
      if (r == 0 || !c.same[r]) { f = 1; s = v; h++; }
      else s += v;
    }
  }
  uint32_t xf, tf;
  uint64_t xs, ts, th;
  block_seg_scan<SCAN_THREADS>(f, s, xf, xs, tf, ts, s_f, s_s);
  block_exclusive_scan_u64(h, s_w, &th);
  if (threadIdx.x == 0) { agg_f[blockIdx.x] = tf; agg_s[blockIdx.x] = ts; heads[blockIdx.x] = th; }
}

// ---- 2. one block: carry[t] = sum of the group that is open where tile t starts (its part in tiles < t)
__global__ void __launch_bounds__(1024) k_comb_carry(const uint32_t *__restrict__ agg_f, const uint64_t *__restrict__ agg_s,
                                                     uint32_t ntiles, uint64_t *__restrict__ carry) {
  __shared__ uint32_t s_f[32];
  __shared__ uint64_t s_s[32];
  uint64_t run = 0;  // flag of the running carry is irrelevant: only its sum is ever used
  for (uint32_t b0 = 0; b0 < ntiles; b0 += 1024) {
    const uint32_t t = b0 + threadIdx.x;
    const uint32_t f = t < ntiles ? agg_f[t] : 0;
    const uint64_t s = t < ntiles ? agg_s[t] : 0;
    uint32_t xf, tf;
    uint64_t xs, ts;
    block_seg_scan<1024>(f, s, xf, xs, tf, ts, s_f, s_s);
    if (t < ntiles) carry[t] = xf ? xs : run + xs;
    run = tf ? ts : run + ts;
  }
}

// ---- 3. apply: the group's head writes (record index, sort word) into the group's slot, its last position the sum
__global__ void __launch_bounds__(SCAN_THREADS)
    k_comb_apply(CombineParams c, const uint32_t *__restrict__ K, const uint64_t *__restrict__ vals,
                 const uint64_t *__restrict__ heads, const uint64_t *__restrict__ carry, uint32_t *__restrict__ g_idx,
                 uint32_t *__restrict__ g_K, uint64_t *__restrict__ g_sum) {
  __shared__ uint32_t s_f[SCAN_THREADS / 32];
  __shared__ uint64_t s_s[SCAN_THREADS / 32], s_w[SCAN_THREADS / 32];
  const uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_IPT;
  uint64_t v[SCAN_IPT];
  uint32_t hd = 0, f = 0, h = 0;  // hd: bit k = position base + k is a group head
  uint64_t s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_IPT; k++) {
    const uint32_t r = base + k;
    v[k] = 0;
    if (r < c.n) {
      v[k] = vals[r];
      if (r == 0 || !c.same[r]) { hd |= 1u << k; f = 1; s = v[k]; h++; }
      else s += v[k];
    }
  }
  uint32_t xf, tf;
  uint64_t xs, ts, th;
  block_seg_scan<SCAN_THREADS>(f, s, xf, xs, tf, ts, s_f, s_s);
  uint64_t g = block_exclusive_scan_u64(h, s_w, &th) + heads[blockIdx.x];  // groups that start before this thread
  uint64_t run = xf ? xs : carry[blockIdx.x] + xs;
#pragma unroll
  for (int k = 0; k < SCAN_IPT; k++) {
    const uint32_t r = base + k;
    if (r >= c.n) break;
    if ((hd >> k) & 1u) {
      run = v[k];
      g_idx[g] = c.order[r];
      g_K[g] = K[r];
      g++;
    } else {
      run += v[k];
    }
    if (r + 1 == c.n || !c.same[r + 1]) g_sum[g - 1] = run;
  }
}

// shortcut path (no two adjacent keys equal): every group is one record, only the value widths need checking
__global__ void k_comb_check_widths(const uint32_t *__restrict__ val_len, uint32_t n, uint32_t vw, uint32_t *__restrict__ bad) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && val_len[i] != vw) atomicMin(bad, i);
}

// ---- pack: group g -> key bytes + big-endian sum.  FIXED: packed at g * (klen + vw); else at off[g] (var mode)
__global__ void k_comb_sizes(Records rec, const uint32_t *__restrict__ g_idx, uint32_t m, uint32_t vw, uint32_t *__restrict__ sizes) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= m) return;
  uint64_t koff;
  uint32_t klen, vlen;
  record_lookup(rec, g_idx[g], koff, klen, vlen);
  sizes[g] = klen + vw;
}

template <bool FIXED>
__global__ void k_comb_pack(Records rec, const uint32_t *__restrict__ g_idx, const uint64_t *__restrict__ g_sum, uint32_t m,
                            uint32_t vw, const uint64_t *__restrict__ off, uint8_t *__restrict__ out, uint32_t *__restrict__ out_klen,
                            uint32_t *__restrict__ out_vlen) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= m) return;
  uint64_t koff;
  uint32_t klen, vlen;
  record_lookup(rec, g_idx[g], koff, klen, vlen);
  uint8_t *d = out + (FIXED ? (uint64_t)g * (klen + vw) : off[g]);
  const uint8_t *k = rec.kv + koff;
  for (uint32_t b = 0; b < klen; b++) d[b] = k[b];
  const uint64_t s = g_sum[g];
  for (uint32_t b = 0; b < vw; b++) d[klen + b] = (uint8_t)(s >> (8 * (vw - 1 - b)));
  if (!FIXED) { out_klen[g] = klen; out_vlen[g] = vw; }
}

__global__ void k_comb_iota(uint32_t *__restrict__ order, uint32_t m) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < m) order[g] = g;
}

}  // namespace tezgpu
