// sorter.cuh -- host orchestration of the device sort pipeline (one "spill" covering everything collected:
// HBM is the sort buffer, so this is always the numSpills==1 branch of PipelinedSorter.flush, :730-756).
#pragma once
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../include/tezgpu.h"
#include "device_util.h"
#ifndef TEZGPU_EMIT_ROUND_FILL_DEFAULT
#define TEZGPU_EMIT_ROUND_FILL_DEFAULT 0
#endif
#include "emit_pipe_u.cuh"
#include "emit_tma.cuh"
#include "emit_runs.cuh"
#include "sorter_kernels.cuh"
#include "combine.cuh"

namespace tezgpu {

// Small device -> host results (flags, counters, the spill index) are WRITTEN BY A KERNEL into mapped pinned memory
// instead of going through cudaMemcpyAsync: a tiny copy is queued on a copy engine, and when another task slot's
// multi-GB upload occupies that engine the sort's one host round trip waits for all of it (measured: a flush next to
// another slot's upload took 297 ms = 144 ms behind the upload + 153 ms of its own; tools/e2e_probe.py).
__global__ void k_store_to_host(uint32_t *__restrict__ dst0, const uint32_t *__restrict__ src0, uint32_t n0, uint32_t *__restrict__ dst1,
                                const uint32_t *__restrict__ src1, uint32_t n1, uint32_t *__restrict__ dst2,
                                const uint32_t *__restrict__ src2, uint32_t n2) {
  for (uint32_t i = threadIdx.x; i < n0; i += blockDim.x) dst0[i] = src0[i];
  for (uint32_t i = threadIdx.x; i < n1; i += blockDim.x) dst1[i] = src1[i];
  for (uint32_t i = threadIdx.x; i < n2; i += blockDim.x) dst2[i] = src2[i];
  __threadfence_system();
}
// up to three word-aligned ranges; dst = cudaHostAlloc memory (device-accessible under unified addressing)
static inline void store_to_host(cudaStream_t st, void *d0, const void *s0, size_t b0, void *d1 = nullptr, const void *s1 = nullptr,
                                 size_t b1 = 0, void *d2 = nullptr, const void *s2 = nullptr, size_t b2 = 0) {
  k_store_to_host<<<1, 256, 0, st>>>((uint32_t *)d0, (const uint32_t *)s0, (uint32_t)(b0 / 4), (uint32_t *)d1, (const uint32_t *)s1,
                                     (uint32_t)(b1 / 4), (uint32_t *)d2, (const uint32_t *)s2, (uint32_t)(b2 / 4));
}


static inline int partition_bits(int P) {
  int b = 0;
  while ((1ll << b) < (long long)P) b++;
  return b;
}

// per-device constant tables (CRC), created once
struct DeviceConstants {
  CrcTables *d_crc = nullptr;
  static DeviceConstants &get(int device) {
    static DeviceConstants inst[64];
    DeviceConstants &d = inst[device & 63];
    if (!d.d_crc) {
      CrcTables *h = new CrcTables();
      crc_build_tables(*h, EMIT_CRC_STRIDE_WORDS);
      TG_CUDA(cudaMalloc((void **)&d.d_crc, sizeof(CrcTables)));
      TG_CUDA(cudaMemcpy(d.d_crc, h, sizeof(CrcTables), cudaMemcpyHostToDevice));
      delete h;
    }
    return d;
  }
};

// thrown by sort_phase in run-table mode (Records::use_runs): the merger then re-parses the segments with the walker
struct FramingMismatch {};

class SortPipeline {
 public:
  tezgpu_conf conf;
  int pbits;
  cudaStream_t stream = nullptr;
  EventTimer timer;
  int num_sms = 148;

  // workspace (grow-only, reused across flushes)
  DeviceBuffer keysA, keysB, valsA, valsB, same, blk, small, tile_state, sizes, rec_off;
  DeviceBuffer t_pos[2], t_gid[2], t_lidx[2], t_key64[2], t_val[2], t_state, t_ghead, t_gneq, sym_sets, sym_tab, rep_flags;
  DeviceBuffer seg_start, tile_start, part_start, d_index, seg_crc, tile_desc, tile_crc, tie_state;
  PinnedBuffer h_small;

  explicit SortPipeline(const tezgpu_conf &c) : conf(c) {
    TG_CHECK(c.num_partitions >= 1, TEZGPU_E_INVALID, "num_partitions must be >= 1");
    TG_CHECK(c.comparator >= TEZGPU_CMP_BYTES && c.comparator <= TEZGPU_CMP_LONG, TEZGPU_E_UNSUPPORTED,
             "comparator outside the device-supported set (BYTES, TEXT, BYTESWRITABLE, INT, LONG)");
    TG_CHECK(c.partitioner == TEZGPU_PART_GIVEN || c.partitioner == TEZGPU_PART_HASH, TEZGPU_E_UNSUPPORTED,
             "partitioner outside the device-supported set (GIVEN, HASH)");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
      cudaGetLastError();
      throw Error(TEZGPU_E_CUDA, "no CUDA device available (libtezgpu has no CPU fallback)");
    }
    TG_CHECK(c.device >= 0 && c.device < ndev, TEZGPU_E_INVALID, "bad device ordinal");
    TG_CUDA(cudaSetDevice(c.device));
    TG_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    TG_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, c.device));
    // The path is dominated by sparse reads (16-byte keys out of 80-byte records, 80-byte record gathers): ask L2 to
    // fetch 32-byte sectors instead of wider granules (measured: stage 1.28 -> 0.70 ms).  TEZGPU_L2_FETCH=0 leaves
    // the device limit untouched, any other value overrides.
    {
      const char *g = getenv("TEZGPU_L2_FETCH");
      int gran = g ? atoi(g) : 32;
      if (gran > 0 && cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)gran) != cudaSuccess) cudaGetLastError();
    }
    pbits = partition_bits(c.num_partitions);
    TG_CHECK(pbits <= 31, TEZGPU_E_INVALID, "too many partitions");
    h_small.ensure(4096);
    small.ensure(16384);
    DeviceConstants::get(c.device);
  }
  ~SortPipeline() {
    if (stream) cudaStreamDestroy(stream);
  }

  static uint64_t output_bound(uint64_t n, uint64_t kv_bytes, int P) { return kv_bytes + 12 * n + 10ull * P + 64; }

  // `small` device scratch layout (u32 words): [0..2047] radix hist (8*256), [2048..2055] trivial flags,
  // [2056..2063] tile counters, [2064] error flag, [2066..2067] dup count (u64), [2068..2071] totals (2 x u64)
  uint32_t *d_hist() { return small.as<uint32_t>(); }
  uint32_t *d_trivial() { return small.as<uint32_t>() + 2048; }
  uint32_t *d_tile_counter() { return small.as<uint32_t>() + 2056; }
  int *d_error() { return reinterpret_cast<int *>(small.as<uint32_t>() + 2064); }
  uint32_t *d_large() { return small.as<uint32_t>() + 2065; }
  uint32_t *d_m() { return small.as<uint32_t>() + 2072; }
  unsigned long long *d_ties() { return reinterpret_cast<unsigned long long *>(small.as<uint32_t>() + 2074); }
  uint32_t *d_ticket() { return small.as<uint32_t>() + 2073; }
  unsigned long long *d_dups() { return reinterpret_cast<unsigned long long *>(small.as<uint32_t>() + 2066); }
  uint64_t *d_totals() { return reinterpret_cast<uint64_t *>(small.as<uint32_t>() + 2068); }

  // state left behind by sort_phase for emit_phase / the merger's record iterator
  struct SortState {
    Records rec;
    uint32_t *K = nullptr;      // sorted sort words
    uint32_t *order = nullptr;  // sorted position -> record index
    uint64_t dup_count = 0, tie_records = 0;
    int launches = 0;
    bool have_bounds = false, spec_layout = false;  // partition bounds / fixed-width layout already on the device
    uint64_t spec_file_bytes = 0, spec_tiles = 0;
    const uint8_t *same = nullptr;  // equal-key flags when they are not the pipeline's own `same` (combined records)
  } state;
  // merge mode only (the Merger sets them): MergeQueue.checkForSameKeys, and "no input record was run-length encoded"
  // (every segment had the plain fixed framing), which together decide whether any record can be written as a repeat
  int merge_check_same = 1;
  bool merge_inputs_plain = false;
  uint32_t merge_max_runs = 0;   // run-table mode: most runs any output partition has (emit_runs.cuh plans <= 32 per warp)
  static bool runs_emit_enabled() {
    // opt-in: measured 8.85 ms per 1e8 records against 8.55 ms for the pipelined gather (emit_pipe_u.cuh), DESIGN.md 7
    static const bool on = getenv("TEZGPU_EMIT_RUNS") && atoi(getenv("TEZGPU_EMIT_RUNS")) != 0;
    return on;
  }

  EmitParams make_emit_params(const Records &rec, const uint32_t *order, int rle, bool merge_mode, uint8_t *d_out) {
    EmitParams e;
    memset(&e, 0, sizeof(e));
    e.rec = rec;
    e.order = order;
    e.same = state.same ? state.same : same.as<uint8_t>();
    e.part_start = part_start.as<uint32_t>();
    e.seg_start = seg_start.as<uint64_t>();
    e.tile_start = tile_start.as<uint32_t>();
    e.out = d_out;
    e.seg_crc = seg_crc.as<uint32_t>();
    e.crc = DeviceConstants::get(conf.device).d_crc;
    e.rle = rle;
    e.send_empty = conf.send_empty_partition_details;
    e.unordered = conf.sorter_impl == TEZGPU_SORTER_UNORDERED;
    e.merge_mode = merge_mode ? 1 : 0;
    e.check_same = merge_check_same;
    e.P = conf.num_partitions;
    return e;
  }
  static bool pipe_unaligned_enabled() {
    // on by default (measured: 9.8 -> 7.9 ms for the 1e8-record reduce-side emit); TEZGPU_EMIT_PIPE_UNALIGNED=0 falls back
    static const bool on = !(getenv("TEZGPU_EMIT_PIPE_UNALIGNED") && atoi(getenv("TEZGPU_EMIT_PIPE_UNALIGNED")) == 0);
    return on;
  }
  void set_fixed_layout(EmitParams &e, const Records &rec) {
    int h = 0;
    for (int b = 0; b < vint_size_u32(rec.klen); b++) e.fixed_hdr[h++] = vint_byte_u32(rec.klen, b);
    for (int b = 0; b < vint_size_u32(rec.vlen); b++) e.fixed_hdr[h++] = vint_byte_u32(rec.vlen, b);
    e.fixed_hdr_len = h;
    e.rec_size = h + rec.klen + rec.vlen;
    // the tile image must fit the image buffer of the source-oriented emit kernels (FE_IMG_BYTES); a record that does
    // not fit it alone (!fast_emit_fits) gets one-record tiles, which the general kernel splits over several images
    e.recs_per_tile = std::max<uint32_t>(1, std::min<uint32_t>(EMIT_MAX_RECS, (FE_IMG_BYTES - 32) / e.rec_size));
    // Round filling: the checksum / write-out loop of the source-oriented kernels walks a tile in rounds of
    // FE_THREADS 16-byte chunks; 256 records of 82 bytes are 5.13 rounds, six are executed.  Among the tile sizes
    // within 10 % of the cap, take the one with the most records per executed round (249 for 82-byte records).
    static const int round_fill = getenv("TEZGPU_EMIT_ROUND_FILL") ? atoi(getenv("TEZGPU_EMIT_ROUND_FILL")) : TEZGPU_EMIT_ROUND_FILL_DEFAULT;
    bool fill = round_fill != 0;
    if (rec.use_runs && runs_emit_enabled() && emit_runs_fits(e.recs_per_tile, e.rec_size, merge_max_runs)) {
      // run-table mode with the range-copy emit (emit_runs.cuh): full 256-record tiles
    } else if (pipe_unaligned_enabled()) {
      // the pipelined kernel for records at arbitrary offsets (emit_pipe_u.cuh) holds a tile's words in five gather rounds
      const uint32_t stride = rec.klen + rec.vlen;
      const bool fast = stride >= 16 && stride % 16 == 0;
      const bool aligned = !rec.key_off && !rec.use_runs && (((uintptr_t)rec.kv & 15u) == 0);
      if (fast && !aligned && emit4u_max_recs(stride / 16) >= 32) {
        e.recs_per_tile = std::min<uint32_t>(e.recs_per_tile, emit4u_max_recs(stride / 16));
        fill = true;
      }
    }
    if (fill && e.recs_per_tile >= 32) {
      const uint32_t cap = e.recs_per_tile;
      uint32_t best = cap;
      double best_eff = 0;
      for (uint32_t r = cap; r >= cap - cap / 10; r--) {
        const uint64_t chunks = ((uint64_t)r * e.rec_size + 15 + 4 + 2 + 15) / 16;  // worst-case lead, header, EOF
        const uint64_t rounds = (chunks + FE_THREADS - 1) / FE_THREADS;
        const double eff = (double)r / (double)rounds;
        if (eff > best_eff) { best_eff = eff; best = r; }
      }
      e.recs_per_tile = best;
    }
    e.rec_off = nullptr;
  }

  void run(Records rec, uint8_t *d_out, uint64_t out_cap, uint64_t *out_len, int64_t *index, tezgpu_stats *stats) {
    sort_phase(rec);
    int rle;
    if (conf.rle_policy == TEZGPU_RLE_ON) rle = 1;
    else if (conf.rle_policy == TEZGPU_RLE_OFF) rle = 0;
    else rle = (conf.sorter_impl == 1) ? 0 : ((double)state.dup_count > 0.1 * (double)rec.n);
    if (conf.sorter_impl == TEZGPU_SORTER_UNORDERED) rle = 0;   // Writer(..., codec, null, null): no run-length encoding (:1092)
    emit_output(rle, false, d_out, out_cap, out_len, index, stats);
  }

  // ---------------- combiner (combine.cuh): TEZGPU_COMBINE_* of the handle; results of the last emit_output
  int combine_kind = TEZGPU_COMBINE_NONE;
  uint64_t combine_in = 0, combine_out = 0;
  float combine_ms = 0;
  DeviceBuffer c_vals, c_aggf, c_aggs, c_heads, c_carry, c_bad, c_idx, c_K, c_sum, c_order, c_same, c_sizes, c_koff, c_klen,
      c_vlen, c_kv;
  EventTimer c_timer;

  // emit_phase of the sorted records, through the combiner when one is set.  The record view of the sort phase is
  // restored afterwards, so the merger's record iterator still walks the uncombined stream.
  void emit_output(int rle, bool merge_mode, uint8_t *d_out, uint64_t out_cap, uint64_t *out_len, int64_t *index,
                   tezgpu_stats *stats) {
    combine_in = combine_out = 0;
    combine_ms = 0;
    if (combine_kind == TEZGPU_COMBINE_NONE) {
      emit_phase(rle, merge_mode, d_out, out_cap, out_len, index, stats);
      return;
    }
    const SortState raw = state;
    const bool combined = combine_phase();
    try {
      emit_phase(rle, merge_mode, d_out, out_cap, out_len, index, stats);
    } catch (...) {
      if (combined) { state = raw; state.have_bounds = state.spec_layout = false; }
      throw;
    }
    if (combined) {
      state = raw;
      state.have_bounds = state.spec_layout = false;  // the emit overwrote the partition bounds and the layout
    }
    if (stats) {
      // OUTPUT_RECORDS and the RLE inputs are counted before the combine, SPILLED_RECORDS / rawLength after it
      stats->output_records = raw.rec.n;
      stats->adjacent_equal_keys = (int64_t)raw.dup_count;
      stats->tie_records = (int64_t)raw.tie_records;
    }
  }

  // Replaces `state` by the combined records (one per group of equal keys, sorted, no two keys equal) and returns true;
  // returns false when the sorted records already are their own combination (no two adjacent keys equal: the sum of one
  // value is that value's bytes).  Value widths are checked either way.
  bool combine_phase() {
    const Records rec = state.rec;
    const uint32_t n = rec.n;
    const uint32_t vw = combine_kind == TEZGPU_COMBINE_INT_SUM ? 4u : 8u;
    const char *what = vw == 4 ? " is not a 4-byte IntWritable" : " is not an 8-byte LongWritable";
    combine_in = combine_out = n;
    if (n == 0) return false;
    if (rec.fixed) TG_CHECK(rec.vlen == vw, TEZGPU_E_INVALID, std::string("combiner value of record 0") + what);
    if (state.dup_count == 0 && rec.fixed) return false;
    c_timer.reset();
    c_timer.mark(stream);
    c_bad.ensure(16);
    TG_CUDA(cudaMemsetAsync(c_bad.p, 0xFF, 4, stream));
    uint32_t *bad = c_bad.as<uint32_t>();
    uint64_t *hs = h_small.as<uint64_t>() + 48;
    auto check_widths = [&]() {
      TG_CUDA(cudaMemcpyAsync(&hs[2], bad, 4, cudaMemcpyDeviceToHost, stream));
      TG_CUDA(cudaStreamSynchronize(stream));
      const uint32_t b = (uint32_t)hs[2];
      TG_CHECK(b == 0xFFFFFFFFu, TEZGPU_E_INVALID, "combiner value of record " + std::to_string(b) + what);
    };
    if (state.dup_count == 0) {
      k_comb_check_widths<<<(uint32_t)div_up(n, 256), 256, 0, stream>>>(rec.val_len, n, vw, bad);
      TG_CUDA(cudaGetLastError());
      check_widths();
      c_timer.mark(stream);
      TG_CUDA(cudaStreamSynchronize(stream));
      combine_ms = c_timer.ms(0, 1);
      return false;
    }
    int launches = state.launches;
    CombineParams cp;
    cp.rec = rec;
    cp.order = state.order;
    cp.same = same.as<uint8_t>();
    cp.n = n;
    cp.vw = vw;
    const uint32_t nblk = (uint32_t)div_up(n, SCAN_TILE);
    c_vals.ensure((size_t)n * 8);
    c_aggf.ensure((size_t)nblk * 4);
    c_aggs.ensure((size_t)nblk * 8);
    c_heads.ensure(((size_t)nblk + 2) * 8);
    c_carry.ensure((size_t)nblk * 8);
    // ---- segmented sum: reduce, scan the tile aggregates and head counts, apply
    k_comb_reduce<<<nblk, SCAN_THREADS, 0, stream>>>(cp, c_vals.as<uint64_t>(), c_aggf.as<uint32_t>(), c_aggs.as<uint64_t>(),
                                                     c_heads.as<uint64_t>(), bad);
    k_scan_block_sums<<<1, 1024, 0, stream>>>(c_heads.as<uint64_t>(), nblk);
    k_comb_carry<<<1, 1024, 0, stream>>>(c_aggf.as<uint32_t>(), c_aggs.as<uint64_t>(), nblk, c_carry.as<uint64_t>());
    launches += 3;
    TG_CUDA(cudaGetLastError());
    TG_CUDA(cudaMemcpyAsync(&hs[0], c_heads.as<uint64_t>() + nblk, 8, cudaMemcpyDeviceToHost, stream));
    check_widths();
    const uint32_t m = (uint32_t)hs[0];
    c_idx.ensure((size_t)m * 4);
    c_K.ensure((size_t)m * 4);
    c_sum.ensure((size_t)m * 8);
    k_comb_apply<<<nblk, SCAN_THREADS, 0, stream>>>(cp, state.K, c_vals.as<uint64_t>(), c_heads.as<uint64_t>(),
                                                    c_carry.as<uint64_t>(), c_idx.as<uint32_t>(), c_K.as<uint32_t>(),
                                                    c_sum.as<uint64_t>());
    launches++;
    // ---- pack the m groups as records in sorted order
    Records cr;
    memset(&cr, 0, sizeof(cr));
    cr.n = m;
    cr.cmp = rec.cmp;
    cr.hash_partition = rec.hash_partition;
    cr.num_partitions = rec.num_partitions;
    cr.pbits = rec.pbits;
    const uint32_t g256 = (uint32_t)div_up(m, 256);
    if (rec.fixed) {
      const uint64_t bytes = (uint64_t)m * (rec.klen + vw);
      c_kv.ensure(bytes + 32);
      k_comb_pack<true><<<g256, 256, 0, stream>>>(rec, c_idx.as<uint32_t>(), c_sum.as<uint64_t>(), m, vw, nullptr,
                                                  c_kv.as<uint8_t>(), nullptr, nullptr);
      launches++;
      cr.fixed = 1;
      cr.klen = rec.klen;
      cr.vlen = vw;
      cr.kv_bytes = bytes;
    } else {
      const uint32_t mblk = (uint32_t)div_up(m, SCAN_TILE);
      c_sizes.ensure((size_t)m * 4);
      c_koff.ensure(((size_t)m + 2) * 8);
      c_klen.ensure((size_t)m * 4);
      c_vlen.ensure((size_t)m * 4);
      blk.ensure(((size_t)mblk + 2) * 8);
      k_comb_sizes<<<g256, 256, 0, stream>>>(rec, c_idx.as<uint32_t>(), m, vw, c_sizes.as<uint32_t>());
      k_sum_u32_blocks<<<mblk, SCAN_THREADS, 0, stream>>>(c_sizes.as<uint32_t>(), m, blk.as<uint64_t>());
      k_scan_block_sums<<<1, 1024, 0, stream>>>(blk.as<uint64_t>(), mblk);
      k_scan_u32_apply<<<mblk, SCAN_THREADS, 0, stream>>>(c_sizes.as<uint32_t>(), m, blk.as<uint64_t>(), c_koff.as<uint64_t>());
      launches += 4;
      TG_CUDA(cudaGetLastError());
      TG_CUDA(cudaMemcpyAsync(&hs[1], c_koff.as<uint64_t>() + m, 8, cudaMemcpyDeviceToHost, stream));
      TG_CUDA(cudaStreamSynchronize(stream));
      const uint64_t bytes = hs[1];
      c_kv.ensure(align_up(bytes, 16) + 32);
      k_comb_pack<false><<<g256, 256, 0, stream>>>(rec, c_idx.as<uint32_t>(), c_sum.as<uint64_t>(), m, vw, c_koff.as<uint64_t>(),
                                                   c_kv.as<uint8_t>(), c_klen.as<uint32_t>(), c_vlen.as<uint32_t>());
      launches++;
      cr.key_off = c_koff.as<uint64_t>();
      cr.key_len = c_klen.as<uint32_t>();
      cr.val_len = c_vlen.as<uint32_t>();
      cr.kv_bytes = align_up(bytes, 16);
    }
    cr.kv = c_kv.as<uint8_t>();
    // identity order, no equal neighbours
    c_order.ensure((size_t)m * 4);
    c_same.ensure(m);
    k_comb_iota<<<g256, 256, 0, stream>>>(c_order.as<uint32_t>(), m);
    TG_CUDA(cudaMemsetAsync(c_same.p, 0, m, stream));
    launches++;
    TG_CUDA(cudaGetLastError());
    c_timer.mark(stream);
    TG_CUDA(cudaStreamSynchronize(stream));
    combine_ms = c_timer.ms(0, 1);
    combine_out = m;
    state.rec = cr;
    state.K = c_K.as<uint32_t>();
    state.order = c_order.as<uint32_t>();
    state.same = c_same.as<uint8_t>();
    state.dup_count = 0;
    state.launches = launches;
    // the partition bounds and the speculative layout of the sort phase describe n records, not m
    state.have_bounds = state.spec_layout = false;
    return true;
  }

  // partition + sort: stage, radix sort of (sort word, index), tie refinement.  Leaves K / order / same / counts.
  void sort_phase(Records rec) {
    TG_CUDA(cudaSetDevice(conf.device));
    const uint32_t n = rec.n;
    const int P = conf.num_partitions;
    TG_CHECK(n <= RADIX_MAX_N, TEZGPU_E_INVALID, "more than 2^30-1 records in one sort");
    rec.cmp = conf.comparator;
    rec.hash_partition = conf.partitioner == TEZGPU_PART_HASH;
    rec.num_partitions = P;
    rec.pbits = pbits;
    const bool unordered = conf.sorter_impl == TEZGPU_SORTER_UNORDERED;
    rec.unordered = unordered ? 1 : 0;
    TG_CHECK(rec.hash_partition || rec.partition || rec.use_runs || n == 0 || P == 1, TEZGPU_E_INVALID, "partition ids required (partitioner=GIVEN)");
    int launches = 0;
    state.have_bounds = state.spec_layout = false;
    timer.reset();
    timer.mark(stream);

    const size_t n4 = (size_t)(n ? n : 1) * 4;
    keysA.ensure(n4); keysB.ensure(n4); valsA.ensure(n4); valsB.ensure(n4);
    same.ensure(n ? n : 1);
    const uint32_t nblk = (uint32_t)div_up(n ? n : 1, SCAN_TILE);
    blk.ensure(((size_t)nblk + 2) * 8);
    part_start.ensure(((size_t)P + 1) * 4);
    seg_start.ensure(((size_t)P + 1) * 8);
    tile_start.ensure(((size_t)P + 1) * 4);
    d_index.ensure((size_t)P * 24);
    seg_crc.ensure((size_t)P * 4);
    h_small.ensure(4096 + (size_t)P * 24);

    TG_CUDA(cudaMemsetAsync(small.p, 0, 16384, stream));
    TG_CUDA(cudaMemsetAsync(seg_crc.p, 0, (size_t)P * 4, stream));

    uint64_t dup_count = 0;
    uint64_t tie_records = 0;
    uint32_t *K = keysA.as<uint32_t>();
    uint32_t *order = valsA.as<uint32_t>();

    uint32_t sym_npos = 0;
    if (n && !rec.fixed && !unordered && !(getenv("TEZGPU_NO_SYM") && atoi(getenv("TEZGPU_NO_SYM")))) {
      // ---------------- alphabet-compressed sort word (SymTable, sorter_kernels.cuh): which byte values occur at the
      // first content positions -> per-position ranks, packed while they fit the (32 - pbits)-bit key field
      sym_sets.ensure(SYM_MAX_POS * 8 * 4);
      sym_tab.ensure(sizeof(SymTable));
      TG_CUDA(cudaMemsetAsync(sym_sets.p, 0, SYM_MAX_POS * 8 * 4, stream));
      k_symbols<<<(int)std::min<uint64_t>(div_up(n, 256), (uint64_t)num_sms * 8), 256, 0, stream>>>(rec, sym_sets.as<uint32_t>());
      launches++;
      uint32_t hs[SYM_MAX_POS * 8];
      TG_CUDA(cudaMemcpyAsync(hs, sym_sets.p, sizeof(hs), cudaMemcpyDeviceToHost, stream));
      TG_CUDA(cudaStreamSynchronize(stream));
      SymTable *t = new SymTable();
      memset(t, 0, sizeof(*t));
      const uint32_t avail = 32u - (uint32_t)pbits;
      uint32_t used = 0, np = 0;
      for (; np < (uint32_t)SYM_MAX_POS; np++) {
        uint32_t cnt = 0;
        for (int w = 0; w < 8; w++) cnt += (uint32_t)__builtin_popcount(hs[np * 8 + w]);
        if (cnt == 0) break;                       // no key is this long
        uint32_t bits = 0;
        while ((1u << bits) < cnt + 1) bits++;     // ranks 1..cnt, 0 = the key ended
        if (used + bits > avail) break;
        used += bits;
        t->shift[np] = (uint8_t)(avail - used);
        uint32_t rk = 0;
        for (uint32_t b = 0; b < 256; b++)
          if ((hs[np * 8 + (b >> 5)] >> (b & 31u)) & 1u) t->rank[np][b] = (uint8_t)(++rk);
      }
      t->npos = np;
      if (np > avail / 8) {                        // packs more positions than the raw bytes would
        TG_CUDA(cudaMemcpyAsync(sym_tab.p, t, sizeof(SymTable), cudaMemcpyHostToDevice, stream));
        TG_CUDA(cudaStreamSynchronize(stream));
        rec.sym = sym_tab.as<SymTable>();
        sym_npos = np;
      }
      delete t;
    }
    if (n) {
      // ---------------- stage
      TG_CUDA(cudaMemsetAsync(same.p, 0, n, stream));
      const bool fast16 = rec.fixed && !rec.key_off && !rec.use_runs && rec.klen == 16 && ((rec.klen + rec.vlen) % 16 == 0) && rec.cmp == CMP_BYTES &&
                          (((uintptr_t)rec.kv & 15u) == 0);
      int sgrid = (int)std::min<uint64_t>(div_up(n, 256), 148 * 16);
      if (fast16) k_stage<true><<<sgrid, 256, 0, stream>>>(rec, K, d_hist(), d_error());
      else k_stage<false><<<sgrid, 256, 0, stream>>>(rec, K, d_hist(), d_error());
      TG_CUDA(cudaGetLastError());
      k_radix_scan_hist<<<1, RADIX, 0, stream>>>(d_hist(), 4, n, d_trivial());
      TG_CUDA(cudaGetLastError());
      launches += 2;
      timer.mark(stream);

      // ---------------- radix sort of (sort word, record index)
      RadixWorkspace ws;
      ws.hist = d_hist();
      ws.trivial = d_trivial();
      ws.tile_counter = d_tile_counter();
      ws.tile_state_words = radix_tile_state_words<uint32_t>(n, 4);
      tile_state.ensure(ws.tile_state_words * 4);
      ws.tile_state = tile_state.as<uint32_t>();
      // unordered: only the passes that cover the partition bits (the top pbits of the word); none when P == 1 -- the
      // first pass is still needed then, to produce the identity index array
      uint32_t pass_mask = 0xF;
      if (unordered) {
        pass_mask = 0;
        for (int q = 0; q < 4; q++) if (8 * q + 8 > 32 - pbits) pass_mask |= 1u << q;
        if (!pass_mask) pass_mask = 1;
      }
      int done = radix_sort_passes<uint32_t>(stream, ws, keysA.as<uint32_t>(), keysB.as<uint32_t>(), valsA.as<uint32_t>(),
                                             valsB.as<uint32_t>(), n, 0, 4, pass_mask, true, &launches);
      if (done & 1) { K = keysB.as<uint32_t>(); order = valsB.as<uint32_t>(); }
      if (unordered) {
        k_flip_order<<<(uint32_t)div_up(n, 256), 256, 0, stream>>>(order, n);
        launches++;
      }
      timer.mark(stream);

      // ---------------- ties: records whose sort words collide are ordered by the rest of the key.
      // One streaming kernel finds the groups and orders the (common) small ones in place; the partition bounds and
      // -- for fixed-width records -- the segment layout are computed speculatively so that the whole common path needs a
      // single host round trip (tie count, large groups, duplicates, error flag, layout totals).
      // normalised content bytes the sort word fully covers (equal words <=> equal on these bytes)
      const uint32_t depth0 = rec.sym ? sym_npos : (uint32_t)((32 - pbits) / 8);
      int per_sm_tf = 0;
      TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_tf, k_tie_fix, TIEFIX_THREADS, 0));
      if (!unordered)   // no comparator on an unordered edge: records of a partition keep their (reversed arrival) order
        k_tie_fix<<<(uint32_t)std::min<uint64_t>(div_up(n, TIEFIX_TILE), (uint64_t)num_sms * std::max(per_sm_tf, 1)), TIEFIX_THREADS, 0, stream>>>(
            rec, K, order, n, depth0, same.as<uint8_t>(), d_dups(), d_large(), d_ties());
      const uint32_t *d_m_ptr = reinterpret_cast<const uint32_t *>(d_ties());
      k_part_bounds<<<(uint32_t)div_up((uint64_t)P + 1, 256), 256, 0, stream>>>(K, n, P, pbits, part_start.as<uint32_t>());
      launches += 2;
      state.have_bounds = true;
      state.spec_layout = false;
      if (rec.fixed) {
        EmitParams e = make_emit_params(rec, order, 0, false, nullptr);
        set_fixed_layout(e, rec);
        k_layout<<<1, 1024, 0, stream>>>(e, seg_start.as<uint64_t>(), tile_start.as<uint32_t>(), d_index.as<int64_t>(), d_totals());
        launches++;
        state.spec_layout = true;
      }
      TG_CUDA(cudaGetLastError());
      uint32_t *hw = h_small.as<uint32_t>();
      store_to_host(stream, hw, small.as<uint32_t>() + 2064, 32, hw + 8, d_m_ptr, 4, h_small.as<uint8_t>() + 4096, d_index.p,
                    state.spec_layout ? (size_t)P * 24 : 0);
      TG_CUDA(cudaGetLastError());
      TG_CUDA(cudaStreamSynchronize(stream));
      // words: [0] error, [1] large groups, [2..3] duplicates, [4..7] layout totals, [8] tied records
      TG_CHECK(!(hw[0] & 1u), TEZGPU_E_INVALID, "Illegal partition (outside [0, numPartitions))");
      if (hw[0] & 2u) throw FramingMismatch();  // run-table mode: some record position lacks the fixed framing bytes
      uint32_t m = hw[8];
      tie_records = m;
      memcpy(&dup_count, hw + 2, 8);
      memcpy(&state.spec_file_bytes, hw + 4, 8);
      memcpy(&state.spec_tiles, hw + 6, 8);
      uint64_t *hs = h_small.as<uint64_t>() + 16;
      if (hw[1]) {
        // some group is larger than TIE_SMALL_MAX: radix refinement rounds over all tied records
        k_tie_count<<<nblk, SCAN_THREADS, 0, stream>>>(K, n, blk.as<uint64_t>());
        k_scan_block_sums<<<1, 1024, 0, stream>>>(blk.as<uint64_t>(), nblk);
        TG_CUDA(cudaMemcpyAsync(&hs[0], blk.as<uint64_t>() + nblk, 8, cudaMemcpyDeviceToHost, stream));
        TG_CUDA(cudaStreamSynchronize(stream));
        m = (uint32_t)hs[0];
        tie_records = m;
        for (int s2 = 0; s2 < 2; s2++) { t_pos[s2].ensure((size_t)m * 4); t_gid[s2].ensure((size_t)m * 4); t_lidx[s2].ensure((size_t)m * 4); }
        k_tie_compact<<<nblk, SCAN_THREADS, 0, stream>>>(K, order, n, blk.as<uint64_t>(), t_pos[0].as<uint32_t>(),
                                                         t_gid[0].as<uint32_t>(), t_lidx[0].as<uint32_t>());
        launches += 3;
        // ---- groups larger than TIE_SMALL_MAX whose members all carry the same key need no ordering (the radix sort
        // is stable): settle them here; only groups with really different keys go through the refinement rounds.
        // Small groups keep the order, flags and duplicate count k_tie_fix gave them.
        const uint32_t ngroups = (uint32_t)(hs[0] >> 32);
        int cur = 0;
        {
          t_ghead.ensure(((size_t)ngroups + 2) * 4);
          t_gneq.ensure((size_t)ngroups + 1);
          TG_CUDA(cudaMemsetAsync(t_gneq.p, 0, (size_t)ngroups + 1, stream));
          const uint32_t mgrid = (uint32_t)div_up(m, 256), mblk0 = (uint32_t)div_up(m, SCAN_TILE);
          k_group_heads<<<mgrid, 256, 0, stream>>>(t_gid[0].as<uint32_t>(), m, t_ghead.as<uint32_t>());
          k_group_equal<<<mgrid, 256, 0, stream>>>(rec, t_gid[0].as<uint32_t>(), t_lidx[0].as<uint32_t>(), t_ghead.as<uint32_t>(), m, depth0,
                                                 TIE_SMALL_MAX, t_gneq.as<uint8_t>());
          blk.ensure(((size_t)std::max(mblk0, nblk) + 2) * 8);
          k_group_mark<<<mblk0, SCAN_THREADS, 0, stream>>>(t_pos[0].as<uint32_t>(), t_gid[0].as<uint32_t>(), t_ghead.as<uint32_t>(),
                                                          t_gneq.as<uint8_t>(), m, TIE_SMALL_MAX, same.as<uint8_t>(), d_dups(), blk.as<uint64_t>());
          k_scan_block_sums<<<1, 1024, 0, stream>>>(blk.as<uint64_t>(), mblk0);
          launches += 4;
          TG_CUDA(cudaGetLastError());
          TG_CUDA(cudaMemcpyAsync(&hs[0], blk.as<uint64_t>() + mblk0, 8, cudaMemcpyDeviceToHost, stream));
          TG_CUDA(cudaStreamSynchronize(stream));
          const uint32_t m2 = (uint32_t)hs[0];
          if (m2) {
            k_group_compact<<<mblk0, SCAN_THREADS, 0, stream>>>(t_pos[0].as<uint32_t>(), t_gid[0].as<uint32_t>(), t_lidx[0].as<uint32_t>(),
                                                               t_ghead.as<uint32_t>(), t_gneq.as<uint8_t>(), m, TIE_SMALL_MAX, blk.as<uint64_t>(),
                                                               t_pos[1].as<uint32_t>(), t_gid[1].as<uint32_t>(), t_lidx[1].as<uint32_t>());
            launches++;
            TG_CUDA(cudaGetLastError());
            cur = 1;
          }
          m = m2;
        }
        uint32_t depth = depth0;
        while (m) {
          t_key64[0].ensure((size_t)m * 8); t_key64[1].ensure((size_t)m * 8); t_val[0].ensure((size_t)m * 4);
          const uint32_t mblk = (uint32_t)div_up(m, SCAN_TILE);
          k_ref_build_keys<<<(uint32_t)div_up(m, 256), 256, 0, stream>>>(rec, t_gid[cur].as<uint32_t>(), t_lidx[cur].as<uint32_t>(), m,
                                                                    depth, t_key64[0].as<uint64_t>());
          TG_CUDA(cudaMemsetAsync(d_hist(), 0, 8 * RADIX * 4, stream));
          k_radix_hist<uint64_t, 8><<<(int)std::min<uint64_t>(div_up(m, 512 * 8), 148 * 4), 512, 0, stream>>>(t_key64[0].as<uint64_t>(), m, 0, d_hist());
          k_radix_scan_hist<<<1, RADIX, 0, stream>>>(d_hist(), 8, m, d_trivial());
          launches += 3;
          TG_CUDA(cudaGetLastError());
          uint32_t *ht = h_small.as<uint32_t>() + 64;
          TG_CUDA(cudaMemcpyAsync(ht, d_trivial(), 8 * 4, cudaMemcpyDeviceToHost, stream));
          TG_CUDA(cudaStreamSynchronize(stream));
          uint32_t mask = 0;
          for (int q = 0; q < 8; q++) if (!ht[q]) mask |= 1u << q;
          RadixWorkspace w2 = ws;
          w2.tile_state_words = radix_tile_state_words<uint64_t>(m, 8);
          t_state.ensure(w2.tile_state_words * 4);
          w2.tile_state = t_state.as<uint32_t>();
          int d2 = radix_sort_passes<uint64_t>(stream, w2, t_key64[0].as<uint64_t>(), t_key64[1].as<uint64_t>(), t_lidx[cur].as<uint32_t>(),
                                               t_val[0].as<uint32_t>(), m, 0, 8, mask, false, &launches);
          const uint64_t *Ks = (d2 & 1) ? t_key64[1].as<uint64_t>() : t_key64[0].as<uint64_t>();
          const uint32_t *Ls = (d2 & 1) ? t_val[0].as<uint32_t>() : t_lidx[cur].as<uint32_t>();
          k_ref_apply_count<<<mblk, SCAN_THREADS, 0, stream>>>(Ks, Ls, t_pos[cur].as<uint32_t>(), m, order, same.as<uint8_t>(), d_dups(),
                                                              blk.as<uint64_t>());
          k_scan_block_sums<<<1, 1024, 0, stream>>>(blk.as<uint64_t>(), mblk);
          launches += 2;
          TG_CUDA(cudaMemcpyAsync(&hs[0], blk.as<uint64_t>() + mblk, 8, cudaMemcpyDeviceToHost, stream));
          TG_CUDA(cudaStreamSynchronize(stream));
          uint32_t m2 = (uint32_t)hs[0];
          if (m2) {
            k_ref_compact<<<mblk, SCAN_THREADS, 0, stream>>>(Ks, Ls, t_pos[cur].as<uint32_t>(), m, blk.as<uint64_t>(),
                                                            t_pos[cur ^ 1].as<uint32_t>(), t_gid[cur ^ 1].as<uint32_t>(),
                                                            t_lidx[cur ^ 1].as<uint32_t>());
            launches++;
            TG_CUDA(cudaGetLastError());
          }
          cur ^= 1;
          m = m2;
          depth += 3;
        }
        TG_CUDA(cudaMemcpyAsync(&hs[0], d_dups(), 8, cudaMemcpyDeviceToHost, stream));
        TG_CUDA(cudaStreamSynchronize(stream));
        dup_count = hs[0];
      }
    }
    timer.mark(stream);
    state.rec = rec;
    state.same = nullptr;
    state.K = K;
    state.order = order;
    state.dup_count = dup_count;
    state.tie_records = tie_records;
    state.launches = launches;
  }

  // layout + emit of the sorted records as IFile segments.  merge_mode: REPEAT_KEY semantics of TezMerger.writeFile
  // (empty keys may be run-length encoded too, SORT/TezMerger.java:215-245).
  void emit_phase(int rle, bool merge_mode, uint8_t *d_out, uint64_t out_cap, uint64_t *out_len, int64_t *index,
                  tezgpu_stats *stats) {
    TG_CUDA(cudaSetDevice(conf.device));
    TG_CHECK(((uintptr_t)d_out & 15u) == 0, TEZGPU_E_INVALID, "output buffer must be 16-byte aligned");
    const Records rec = state.rec;
    const uint32_t n = rec.n;
    const int P = conf.num_partitions;
    uint32_t *K = state.K, *order = state.order;
    const uint64_t dup_count = state.dup_count, tie_records = state.tie_records;
    int launches = state.launches;
    const CrcTables *d_crc = DeviceConstants::get(conf.device).d_crc;
    const size_t n4 = (size_t)(n ? n : 1) * 4;
    const uint32_t nblk = (uint32_t)div_up(n ? n : 1, SCAN_TILE);
    TG_CUDA(cudaMemsetAsync(seg_crc.p, 0, (size_t)P * 4, stream));
    if (timer.n > (n ? 4 : 2)) timer.n = n ? 4 : 2;  // re-emit: drop the marks of a previous emit

    // ---------------- layout + emit
    EmitParams e = make_emit_params(rec, order, rle, merge_mode, d_out);
    if (!state.have_bounds) {
      k_part_bounds<<<(uint32_t)div_up((uint64_t)P + 1, 256), 256, 0, stream>>>(K, n, P, pbits, part_start.as<uint32_t>());
      launches++;
    }
    // constant-size framing is only valid when no record is written as a repeat (merge mode flags repeats on its own)
    // (a merge writes repeats for isSameKey() records: none exist when checkForSameKeys is off and no input was encoded)
    const bool no_repeats = !rle && (!merge_mode || (!merge_check_same && merge_inputs_plain));
    const bool fixed_emit = rec.fixed && (dup_count == 0 || no_repeats);
    uint64_t bound = output_bound(n, rec.fixed ? (uint64_t)n * (rec.klen + rec.vlen) : rec.kv_bytes, P);
    uint64_t *hs = h_small.as<uint64_t>();
    if (fixed_emit && state.spec_layout) {
      // layout, totals and index triples were produced during the sort phase (same parameters): no round trip here
      set_fixed_layout(e, rec);
      hs[0] = state.spec_file_bytes;
      hs[1] = state.spec_tiles;
    } else {
      if (fixed_emit) {
        set_fixed_layout(e, rec);
      } else {
        uint64_t avg = n ? (rec.fixed ? (uint64_t)(rec.klen + rec.vlen) : rec.kv_bytes / n) + 4 : 16;
        e.recs_per_tile = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(EMIT_MAX_RECS, (EMIT_IMG_BYTES - 32) / avg));
        sizes.ensure(n4);
        rec_off.ensure(((size_t)n + 2) * 8);
        if (n) {
          rep_flags.ensure(n);
          k_emit_repeat_flags<<<(uint32_t)div_up(n, 256), 256, 0, stream>>>(e, K, rep_flags.as<uint8_t>());
          launches++;
          e.rep = rep_flags.as<uint8_t>();
          k_emit_sizes<<<(uint32_t)div_up(n, 256), 256, 0, stream>>>(e, K, sizes.as<uint32_t>());
          k_sum_u32_blocks<<<nblk, SCAN_THREADS, 0, stream>>>(sizes.as<uint32_t>(), n, blk.as<uint64_t>());
          k_scan_block_sums<<<1, 1024, 0, stream>>>(blk.as<uint64_t>(), nblk);
          k_scan_u32_apply<<<nblk, SCAN_THREADS, 0, stream>>>(sizes.as<uint32_t>(), n, blk.as<uint64_t>(), rec_off.as<uint64_t>());
          launches += 4;
          TG_CUDA(cudaGetLastError());
        } else {
          TG_CUDA(cudaMemsetAsync(rec_off.p, 0, 16, stream));
        }
        e.rec_off = rec_off.as<uint64_t>();
      }
      k_layout<<<1, 1024, 0, stream>>>(e, seg_start.as<uint64_t>(), tile_start.as<uint32_t>(), d_index.as<int64_t>(), d_totals());
      launches++;
      TG_CUDA(cudaGetLastError());
      store_to_host(stream, &hs[0], d_totals(), 16, h_small.as<uint8_t>() + 4096, d_index.p, (size_t)P * 24);
      TG_CUDA(cudaGetLastError());
      TG_CUDA(cudaStreamSynchronize(stream));
      state.spec_layout = false;  // the device layout now belongs to this emit
    }
    const uint64_t file_bytes = hs[0];
    const uint64_t tiles = hs[1];
    TG_CHECK(file_bytes <= bound, TEZGPU_E_INVALID, "internal: output exceeds bound");
    TG_CHECK(file_bytes <= out_cap, TEZGPU_E_NOMEM, "output buffer too small for file.out");
    // fixed-width records take the source-oriented kernel (emit_fast.cuh): 16-byte aligned packed records use one
    // 128-bit load per piece, records at explicit / unaligned offsets two loads + a funnel shift
    const uint32_t stride = rec.klen + rec.vlen;
    const bool fast_emit = fixed_emit && stride >= 16 && (stride % 16 == 0) && fast_emit_fits(e.rec_size) &&
                           !getenv("TEZGPU_NO_FAST_EMIT");
    const bool fast_aligned = fast_emit && !rec.key_off && !rec.use_runs && (((uintptr_t)rec.kv & 15u) == 0);
    FastEmitParams fp;
    if (tiles && fast_emit) {
      tile_desc.ensure((size_t)tiles * sizeof(TileDesc));
      k_build_tiles<<<(uint32_t)div_up(tiles, 256), 256, 0, stream>>>(e, tile_desc.as<TileDesc>());
      launches++;
      fp.e = e;
      tile_crc.ensure((size_t)tiles * sizeof(TileCrc));
      fp.tile_crc = tile_crc.as<TileCrc>();
      fp.tiles = tile_desc.as<TileDesc>();
      fp.ntiles = (uint32_t)tiles;
      fp.cpr = stride / 16;
      fp.cpr_magic = fp.cpr == 1 ? 0u : (uint32_t)((1ull << 32) / fp.cpr) + 1u;
      fp.stride = stride;
    }
    timer.mark(stream);
    if (tiles) {
      if (fast_emit) {
        int per_sm = 0;
        // opt-in (TEZGPU_EMIT_TMA=1): byte-exact (68 GPU parity tests), but measured 15.4 ms against 5.45 ms for the
        // register-staged kernel on 1e8 records -- the bulk-copy gather itself is as fast as the LDG gather
        // (tools/bench_gather.cu: 4.4 ms either way, the memory system's rate for random 80-byte reads), the warp-divergent
        // chunk assembly of the consumers is what costs (profiles/README.md, round 2)
        static const bool use_tma = getenv("TEZGPU_EMIT_TMA") && atoi(getenv("TEZGPU_EMIT_TMA")) != 0;
        if (fast_aligned && use_tma && emit_tma_fits(e.recs_per_tile, stride)) {
          // gather by the bulk-copy engine into a shared-memory ring, chunks assembled straight from the staged
          // records (emit_tma.cuh); TEZGPU_EMIT_TMA=0 selects the register-staged kernels below
          const size_t smem = EmitTmaLayout::total(e.recs_per_tile, stride);
          static size_t attr_smem = 0;
          if (smem > attr_smem) {
            TG_CUDA(cudaFuncSetAttribute(k_emit_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_smem = smem;
          }
          TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_emit_tma, ET_THREADS, smem));
          uint32_t grid = (uint32_t)std::min<uint64_t>(tiles, (uint64_t)num_sms * (per_sm > 0 ? per_sm : 1));
          k_emit_tma<<<grid, ET_THREADS, smem, stream>>>(fp, (uint32_t)EmitTmaLayout::stage_bytes(e.recs_per_tile, stride));
        } else if (fast_aligned && emit4_fits(e.recs_per_tile, fp.cpr) && !getenv("TEZGPU_EMIT_V2")) {
          // software-pipelined kernel (emit_pipe.cuh): a tile's pieces must fit one stage of its gather ring.
          // Default: independent 256-thread CTAs, three per SM.  TEZGPU_EMIT_SUBS=3 selects the variant with one CTA
          // per SM whose three groups share lane-private checksum tables -- measured SLOWER (8.39 vs 5.44 ms): its
          // 219 KB of shared memory leave the SM ~30 KB of L1 and the random gather loses its memory-level parallelism.
          static const bool subs1 = !(getenv("TEZGPU_EMIT_SUBS") && atoi(getenv("TEZGPU_EMIT_SUBS")) == 3);
          if (!subs1) {
            constexpr int SUBS = 3;
            static bool attr = false;
            if (!attr) {
              TG_CUDA(cudaFuncSetAttribute(k_emit_fast4<FE4_UNROLL, SUBS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Emit4Smem<SUBS>::TOTAL));
              attr = true;
            }
            uint32_t grid = (uint32_t)std::min<uint64_t>(div_up(tiles, SUBS), (uint64_t)num_sms);
            k_emit_fast4<FE4_UNROLL, SUBS><<<grid, FE_THREADS * SUBS, Emit4Smem<SUBS>::TOTAL, stream>>>(fp);
          } else {
            static bool attr = false;
            if (!attr) {
              TG_CUDA(cudaFuncSetAttribute(k_emit_fast4<FE4_UNROLL, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Emit4Smem<1>::TOTAL));
              attr = true;
            }
            TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_emit_fast4<FE4_UNROLL, 1>, FE_THREADS, Emit4Smem<1>::TOTAL));
            uint32_t grid = (uint32_t)std::min<uint64_t>(tiles, (uint64_t)num_sms * (per_sm > 0 ? per_sm : 1));
            k_emit_fast4<FE4_UNROLL, 1><<<grid, FE_THREADS, Emit4Smem<1>::TOTAL, stream>>>(fp);
          }
        } else if (rec.use_runs && runs_emit_enabled() && emit_runs_fits(e.recs_per_tile, e.rec_size, merge_max_runs)) {
          // reduce side, fixed-framing runs in place: one bulk copy per run and tile (emit_runs.cuh)
          const size_t smem = EmitRunsLayout::total(e.recs_per_tile, e.rec_size);
          static size_t attr_smem = 0;
          if (smem > attr_smem) {
            TG_CUDA(cudaFuncSetAttribute(k_emit_runs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_smem = smem;
          }
          TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_emit_runs, ER_THREADS, smem));
          uint32_t grid = (uint32_t)std::min<uint64_t>(tiles, (uint64_t)num_sms * (per_sm > 0 ? per_sm : 1));
          k_emit_runs<<<grid, ER_THREADS, smem, stream>>>(fp, (uint32_t)EmitRunsLayout::stage_data(e.recs_per_tile, e.rec_size),
                                                         (uint32_t)EmitRunsLayout::stage_bytes(e.recs_per_tile, e.rec_size));
        } else if (fast_aligned) {
          TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_emit_fast<5, true>, FE_THREADS, 0));
          uint32_t grid = (uint32_t)std::min<uint64_t>(tiles, (uint64_t)num_sms * (per_sm > 0 ? per_sm : 1));
          k_emit_fast<5, true><<<grid, FE_THREADS, 0, stream>>>(fp);
        } else if (!fast_aligned && pipe_unaligned_enabled() && e.recs_per_tile <= emit4u_max_recs(fp.cpr)) {
          // records at arbitrary offsets (reduce side), software-pipelined variant
          static bool attr = false;
          if (!attr) {
            TG_CUDA(cudaFuncSetAttribute(k_emit_fast4u<FE4U_UNROLL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Emit4uSmem::TOTAL));
            attr = true;
          }
          TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_emit_fast4u<FE4U_UNROLL>, FE_THREADS, Emit4uSmem::TOTAL));
          uint32_t grid = (uint32_t)std::min<uint64_t>(tiles, (uint64_t)num_sms * (per_sm > 0 ? per_sm : 1));
          k_emit_fast4u<FE4U_UNROLL><<<grid, FE_THREADS, Emit4uSmem::TOTAL, stream>>>(fp);
        } else {
          TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_emit_fast<5, false>, FE_THREADS, 0));
          uint32_t grid = (uint32_t)std::min<uint64_t>(tiles, (uint64_t)num_sms * (per_sm > 0 ? per_sm : 1));
          k_emit_fast<5, false><<<grid, FE_THREADS, 0, stream>>>(fp);
        }
        k_crc_combine<<<(uint32_t)div_up(tiles, 256), 256, 0, stream>>>(fp.tile_crc, (uint32_t)tiles, d_crc, seg_crc.as<uint32_t>());
        launches++;
      } else {
        // general kernel, persistent CTAs (as many as fit the device at once)
        static int per_sm_fixed = 0, per_sm_var = 0;
        if (!per_sm_fixed) {
          TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_fixed, k_emit<true>, EMIT_THREADS, 0));
          TG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_var, k_emit<false>, EMIT_THREADS, 0));
        }
        const uint32_t cap = (uint32_t)num_sms * (uint32_t)std::max(1, fixed_emit ? per_sm_fixed : per_sm_var);
        const uint32_t grid = (uint32_t)std::min<uint64_t>(tiles, cap);
        if (fixed_emit) k_emit<true><<<grid, EMIT_THREADS, 0, stream>>>(e);
        else k_emit<false><<<grid, EMIT_THREADS, 0, stream>>>(e);
      }
      launches++;
      TG_CUDA(cudaGetLastError());
    }
    timer.mark(stream);
    k_finalize_segments<<<(uint32_t)div_up(P, 256), 256, 0, stream>>>(e);
    launches++;
    TG_CUDA(cudaGetLastError());
    timer.mark(stream);
    TG_CUDA(cudaStreamSynchronize(stream));

    if (out_len) *out_len = file_bytes;
    const int64_t *hidx = reinterpret_cast<const int64_t *>(h_small.as<uint8_t>() + 4096);
    if (index) memcpy(index, hidx, (size_t)P * 24);
    if (stats) {
      memset(stats, 0, sizeof(*stats));
      stats->output_records = n;
      int64_t raw = 0;
      for (int p = 0; p < P; p++) raw += hidx[3 * p + 1];
      stats->output_bytes_with_overhead = raw;
      stats->output_bytes_physical = (int64_t)file_bytes;
      stats->file_out_bytes = (int64_t)file_bytes;
      stats->spilled_records = n;
      stats->num_spills = 1;
      stats->rle_used = rle;
      stats->adjacent_equal_keys = (int64_t)dup_count;
      stats->tie_records = (int64_t)tie_records;
      // marks: n>0: start, stage, sort, ties, pre-emit-kernel, post-emit-kernel, end ; n==0: start, ties, pre, post, end
      const int b = n ? 3 : 1;
      stats->ms_stage = n ? timer.ms(0, 1) : 0;
      stats->ms_sort = n ? timer.ms(1, 2) : 0;
      stats->ms_ties = n ? timer.ms(2, 3) : 0;
      stats->ms_emit = timer.ms(b, b + 3);
      stats->ms_emit_kernel = timer.ms(b + 1, b + 2);
      stats->ms_total = timer.ms(0, b + 3);
      stats->kernel_launches = launches;
    }
  }
};

}  // namespace tezgpu
