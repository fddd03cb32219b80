// merger.cuh -- reduce side of the hot path on sm_100a: k-way merge of sorted IFile segments.
// Device counterpart of TezMerger.MergeQueue (SORT/TezMerger.java:465-1065): segments are checksum-verified and
// parsed on the device, the union of their records is ordered with the same radix-sort + key-refinement machinery
// as the map side (a stable sort of already sorted runs IS their k-way merge: equal keys keep (segment, position)
// order), and the merged stream is either iterated (TezRawKeyValueIterator) or written as one IFile segment
// (TezMerger.writeFile, :215-245) with REPEAT_KEY run-length encoding of equal adjacent keys.
#pragma once
#include <algorithm>
#include <vector>

#include "sorter.cuh"
#include "parse_windows.cuh"

namespace tezgpu {

struct SegDesc {
  uint64_t off;       // offset of the segment in the staging buffer (16-byte aligned)
  uint64_t len;       // total bytes
  uint64_t body0;     // offset of the first body byte inside the segment (4 with header, 0 in-memory)
  uint64_t body_end;  // offset just past the EOF markers' possible position: len - 4 (checksum / slack excluded)
  uint32_t has_header;  // bit 0: 'TIF' header present; bit 1: checksum already verified by the transport (skip)
  uint32_t partition;
};

// ------------------------------------------------------------------------------------------------ checksum
// raw CRC remainder of 64 KiB pieces of the segment bodies, combined per segment by k_crc_combine
constexpr uint32_t CRC_PIECE = 64 * 1024;
constexpr int CRCV_THREADS = 256;

__global__ void __launch_bounds__(CRCV_THREADS)
    k_crc_pieces(const uint8_t *__restrict__ data, const SegDesc *__restrict__ segs, const uint32_t *__restrict__ piece_start,
                 uint32_t nseg, const CrcTables *__restrict__ t, TileCrc *__restrict__ out) {
  static_assert(CRCV_THREADS == EMIT_CRC_STRIDE_WORDS, "advc is built for this chunk interleave");
  __shared__ uint32_t s_tab[256], s_adv128[4 * 256], s_part[CRCV_THREADS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  s_tab[tid] = t->slice[0][tid];
  for (int i = tid; i < 4 * 256; i += CRCV_THREADS) s_adv128[i] = (&t->adv128[0][0])[i];
  // the two maps of the 16-byte-chunk interleave as warp-resident digit tables (crc32.cuh)
  CrcChunkFoldT<true> cf;
  cf.init(t, lane);
  const uint32_t piece = blockIdx.x;
  uint32_t lo = 0, hi = nseg;  // last segment with piece_start[s] <= piece
  while (hi - lo > 1) {
    uint32_t mid = (lo + hi) >> 1;
    if (piece_start[mid] <= piece) lo = mid; else hi = mid;
  }
  const SegDesc sd = segs[lo];
  const uint64_t body_bytes = sd.body_end - sd.body0;
  const uint64_t a = (uint64_t)(piece - piece_start[lo]) * CRC_PIECE;
  const uint64_t b = min(body_bytes, a + CRC_PIECE);
  // piece = body bytes [a, b) seen as 16-byte chunks from the aligned-down address: bytes of the first chunk that
  // precede the piece are masked to zero (a remainder with zero initial value ignores leading zeros), the trailing
  // partial chunk is folded bytewise by lane 0.  Thread t owns the chunks whose distance from the last whole chunk is
  // == T-1-t (mod T): 3 x "next word" and one "skip to my next chunk" per chunk, partials aligned by a constant.
  const uint8_t *base = data + sd.off + sd.body0;
  const uint8_t *pa = base + a, *pb = base + b;
  const uint32_t mis = (uint32_t)((uintptr_t)pa & 15u);
  const uint4 *c16 = reinterpret_cast<const uint4 *>(pa - mis);
  const uint32_t Cn = (uint32_t)((pb - (pa - mis)) >> 4);  // whole chunks
  uint32_t c = 0;
  if (Cn) {
    const uint32_t iters = (Cn + CRCV_THREADS - 1) / CRCV_THREADS;
    const int32_t last_i = (int32_t)Cn - CRCV_THREADS + tid;
    int32_t i = last_i - (int32_t)(iters - 1) * CRCV_THREADS;
    for (uint32_t it = 0; it < iters; it++, i += CRCV_THREADS) {
      uint4 v = make_uint4(0, 0, 0, 0);
      if (i >= 0) {
        v = c16[i];
        if (i == 0 && mis) {
          uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (uint32_t k = 0; k < 4; k++) {
            if (mis >= 4 * k + 4) w[k] = 0;
            else if (mis > 4 * k) w[k] &= 0xFFFFFFFFu << (8u * (mis - 4 * k));
          }
          v = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
      c = cf.fold(c, v, it + 1 == iters);
    }
  }
  s_part[tid] = c;
  __syncthreads();
  if (warp == 0) {
    // lane l folds partials l, l+32, ... (Horner with x^(128*32)), aligns by x^(128*(31-l)), xor-reduce
    uint32_t q = 0;
#pragma unroll
    for (int k = 0; k < CRCV_THREADS / 32; k++) {
      q = s_adv128[q & 0xFF] ^ s_adv128[256 + ((q >> 8) & 0xFF)] ^ s_adv128[512 + ((q >> 16) & 0xFF)] ^ s_adv128[768 + (q >> 24)];
      q ^= s_part[lane + 32 * k];
    }
    q = crc_multmodp(q, cf.lane_pow);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) q ^= __shfl_xor_sync(0xffffffffu, q, o);
    if (lane == 0) {
      uint32_t raw = q;
      const uint8_t *tail = Cn ? (pa - mis) + 16ull * Cn : pa;  // no whole chunk: everything bytewise
      for (const uint8_t *x = tail; x < pb; x++) raw = s_tab[(raw ^ *x) & 0xFF] ^ (raw >> 8);
      TileCrc tc;
      tc.raw = raw;
      tc.p = lo;
      tc.after = body_bytes - b;
      out[piece] = tc;
    }
  }
}

// verifyHeaderMagic + compressed flag (SORT/IFile.java:1004-1016): 1 = bad magic, 2 = compressed segment
__global__ void k_check_headers(const uint8_t *__restrict__ data, const SegDesc *__restrict__ segs, uint32_t nseg,
                                int *__restrict__ bad_magic, int *__restrict__ compressed) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  const SegDesc sd = segs[s];
  if (!(sd.has_header & 1u)) return;
  const uint8_t *h = data + sd.off;
  if (!(h[0] == 'T' && h[1] == 'I' && h[2] == 'F')) atomicExch(bad_magic, (int)s + 1);
  else if (h[3] != 0) atomicExch(compressed, (int)s + 1);
}

// compares the folded remainder with the big-endian trailer (SORT/IFileInputStream.java:235-289)
__global__ void k_crc_check(const uint8_t *__restrict__ data, const SegDesc *__restrict__ segs, uint32_t nseg,
                            const uint32_t *__restrict__ seg_crc, const CrcTables *__restrict__ t, int *__restrict__ bad) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  const SegDesc sd = segs[s];
  // in-memory segments carry no checksum stream (OG/InMemoryReader.java:142-254); segments the transport verified
  // while copying them (IFile.Reader.readToMemory, SORT/IFile.java:764-809) are not verified twice
  if (sd.has_header != 1u) return;
  const uint64_t body = sd.body_end - sd.body0;
  uint32_t crc = seg_crc[s] ^ crc_shift_bytes(t, 0xFFFFFFFFu, body) ^ 0xFFFFFFFFu;
  const uint8_t *tr = data + sd.off + sd.body_end;
  uint32_t stored = ((uint32_t)tr[0] << 24) | ((uint32_t)tr[1] << 16) | ((uint32_t)tr[2] << 8) | tr[3];
  if (crc != stored) atomicExch(bad, (int)s + 1);
}

// ------------------------------------------------------------------------------------------------ parse
// hadoop WritableUtils.readVLong with bounds; returns false when the buffer ends inside the vint
__device__ __forceinline__ bool read_vlong_dev(const uint8_t *p, uint64_t &pos, uint64_t end, int64_t &out) {
  if (pos >= end) return false;
  int8_t first = (int8_t)p[pos];
  int len = vint_decode_size((uint8_t)first);
  if (pos + (uint64_t)len > end) return false;
  if (len == 1) { out = first; pos += 1; return true; }
  uint64_t v = 0;
  for (int i = 1; i < len; i++) v = (v << 8) | p[pos + i];
  bool neg = first < -120 || (first >= -112 && first < 0);
  out = neg ? (int64_t)~v : (int64_t)v;
  pos += len;
  return true;
}

struct ParseArrays {
  uint64_t *key_off;
  uint64_t *val_off;
  uint32_t *key_len;
  uint32_t *val_len;
  uint32_t *tag;  // (segment << 1) | read as SAME_KEY (run-length encoded in the input)
  int32_t *partition;
};

// Walks the segments with IFile.Reader semantics (positionToNextRecord / readRawKey / nextRawValue,
// SORT/IFile.java:877-1000).  One WARP per segment: the 32 lanes stage a 4 KiB window of the body in shared memory with
// coalesced loads, lane 0 decodes the record headers out of it (key / value bytes are skipped, never read), so a walk
// step costs tens of cycles instead of a DRAM round trip.  EMIT=false counts records, EMIT=true writes their metadata
// at rec_base[s]...
constexpr int PARSE_WARPS = 8;
constexpr uint32_t PARSE_WIN = 4096;

struct ParseWin {
  const uint8_t *seg;   // segment base in global memory
  uint8_t *win;         // this warp's shared window
  uint64_t wbase;       // segment offset of win[0]
  uint64_t end;         // body end
};
// byte of the segment at offset pos; returns false when pos is outside the staged window (caller reloads)
__device__ __forceinline__ bool pw_byte(const ParseWin &w, uint64_t pos, uint8_t &out) {
  if (pos < w.wbase || pos >= w.wbase + PARSE_WIN) return false;
  out = w.win[pos - w.wbase];
  return true;
}
// readVLong from the window: 0 = ok, 1 = need reload at pos, 2 = runs past the body end
__device__ __forceinline__ int pw_vlong(const ParseWin &w, uint64_t &pos, int64_t &out) {
  if (pos >= w.end) return 2;
  uint8_t first;
  if (!pw_byte(w, pos, first)) return 1;
  const int len = vint_decode_size(first);
  if (pos + (uint64_t)len > w.end) return 2;
  if (pos + (uint64_t)len > w.wbase + PARSE_WIN) return 1;
  if (len == 1) { out = (int8_t)first; pos += 1; return 0; }
  uint64_t v = 0;
  for (int i = 1; i < len; i++) v = (v << 8) | w.win[pos + i - w.wbase];
  const int8_t f = (int8_t)first;
  const bool neg = f < -120 || (f >= -112 && f < 0);
  out = neg ? (int64_t)~v : (int64_t)v;
  pos += len;
  return 0;
}

template <bool EMIT>
__global__ void __launch_bounds__(PARSE_WARPS * 32)
    k_parse_segments(const uint8_t *__restrict__ data, const SegDesc *__restrict__ segs, uint32_t nseg,
                     uint64_t *__restrict__ counts /*[nseg] records*/, uint64_t *__restrict__ kvbytes /*[nseg]*/,
                     const uint64_t *__restrict__ rec_base, ParseArrays out, int *__restrict__ bad) {
  __shared__ __align__(16) uint8_t s_win[PARSE_WARPS][PARSE_WIN];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t s = blockIdx.x * PARSE_WARPS + warp;
  if (s >= nseg) return;
  const SegDesc sd = segs[s];
  ParseWin w;
  w.seg = data + sd.off;
  w.win = s_win[warp];
  w.end = sd.body_end;
  w.wbase = sd.body0;
  // walker state (lane 0)
  uint64_t pos = sd.body0;
  int64_t cur_klen = 0, cur_vlen = 0;
  uint64_t orig_koff = 0;
  int64_t orig_klen = 0;
  uint64_t n = 0, bytes = 0;
  const uint64_t base = EMIT ? rec_base[s] : 0;
  int status = 0;  // 0 running, 1 done ok, 2 malformed
  int phase = 0;   // resume point inside a record: 0 = lengths not read yet
  while (true) {
    // ---- stage the window [wbase, wbase + WIN) (clamped to the segment) with coalesced loads
    {
      const uint64_t seg_len = sd.len;
      for (uint32_t o = lane * 4; o < PARSE_WIN; o += 128) {
        const uint64_t p = w.wbase + o;
        uint32_t v = 0;
        if (p + 4 <= seg_len && (((uintptr_t)(w.seg + p)) & 3u) == 0) v = *reinterpret_cast<const uint32_t *>(w.seg + p);
        else for (int b = 0; b < 4; b++) if (p + b < seg_len) v |= (uint32_t)w.seg[p + b] << (8 * b);
        *reinterpret_cast<uint32_t *>(w.win + o) = v;
      }
    }
    __syncwarp();
    if (lane == 0) {
      while (status == 0) {
        // record lengths (restartable: nothing is committed until all vints of the record header are decoded)
        uint64_t p2 = pos;
        int64_t kl = cur_klen, vl = cur_vlen;
        int rc;
        if (cur_klen == -2) {  // previous record was a repeat: a value length (or V_END_MARKER + both lengths) follows
          rc = pw_vlong(w, p2, vl);
          if (rc == 0 && vl == -3) { rc = pw_vlong(w, p2, kl); if (rc == 0) rc = pw_vlong(w, p2, vl); }
        } else {
          rc = pw_vlong(w, p2, kl);
          if (rc == 0) rc = pw_vlong(w, p2, vl);
        }
        if (rc == 1) { w.wbase = pos & ~(uint64_t)15; break; }  // reload the window at the record start
        if (rc == 2) { status = 2; break; }
        if (kl == -1 && vl == -1) { status = 1; break; }           // EOF markers
        if ((kl != -2 && kl < 0) || vl < 0 || kl > 0x7fffffffll || vl > 0x7fffffffll) { status = 2; break; }
        pos = p2;
        cur_klen = kl;
        cur_vlen = vl;
        if (kl != -2) {
          if (pos + (uint64_t)kl > w.end) { status = 2; break; }
          orig_koff = pos;
          orig_klen = kl;
          pos += (uint64_t)kl;
        } else if (n == 0) { status = 2; break; }  // a repeat needs a previous key
        if (pos + (uint64_t)vl > w.end) { status = 2; break; }
        if (EMIT) {
          // a repeated key points at the bytes of the last full key; its value bytes are not adjacent to it
          out.key_off[base + n] = sd.off + orig_koff;
          out.val_off[base + n] = sd.off + pos;
          out.key_len[base + n] = (uint32_t)orig_klen;
          out.val_len[base + n] = (uint32_t)vl;
          out.tag[base + n] = (s << 1) | (kl == -2 ? 1u : 0u);
          out.partition[base + n] = (int32_t)sd.partition;
        }
        n++;
        bytes += (uint64_t)orig_klen + (uint64_t)vl;
        pos += (uint64_t)vl;
      }
    }
    (void)phase;
    status = __shfl_sync(0xffffffffu, status, 0);
    w.wbase = __shfl_sync(0xffffffffu, w.wbase, 0);
    if (status != 0) break;
    __syncwarp();
  }
  if (lane == 0) {
    if (status == 2) atomicExch(bad, (int)s + 1);
    if (!EMIT) { counts[s] = n; kvbytes[s] = bytes; }
  }
}

// run-table mode -> explicit arrays (only when the record iterator or the run-length encoding emit needs them):
// every body is exactly n records of a known framing (checked by k_stage), so the metadata is pure arithmetic
__global__ void k_fill_fixed_arrays(const SegDesc *__restrict__ segs, uint32_t nseg, const uint64_t *__restrict__ rec_base,
                                    uint32_t klen, uint32_t vlen, uint32_t hdr_len, ParseArrays out) {
  const uint64_t total = rec_base[nseg];
  const uint32_t rs = hdr_len + klen + vlen;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t lo = 0, hi = nseg;  // segment of record i
    while (hi - lo > 1) {
      uint32_t mid = (lo + hi) >> 1;
      if (rec_base[mid] <= i) lo = mid; else hi = mid;
    }
    const SegDesc sd = segs[lo];
    const uint64_t pos = sd.off + sd.body0 + (i - rec_base[lo]) * rs;
    out.key_off[i] = pos + hdr_len;
    out.val_off[i] = pos + hdr_len + klen;
    out.key_len[i] = klen;
    out.val_len[i] = vlen;
    out.tag[i] = lo << 1;
    out.partition[i] = (int32_t)sd.partition;
  }
}

// ------------------------------------------------------------------------------------------------ iterator batches
// kv_off[r] = sum of (klen + vlen) of the merged records before sorted position r
__global__ void __launch_bounds__(256) k_kv_sizes(Records rec, const uint32_t *__restrict__ order, uint32_t *__restrict__ sizes) {
  uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rec.n) return;
  uint32_t i = order[r];
  sizes[r] = rec.key_len[i] + rec.val_len[i];
}

// largest count <= max_records starting at `cursor` whose key+value bytes fit in cap
__global__ void k_find_batch(const uint64_t *__restrict__ kv_off, uint32_t n, uint32_t cursor, uint32_t max_records,
                             uint64_t cap, uint32_t *__restrict__ out_count) {
  uint32_t lo = 0, hi = min(max_records, n - cursor);
  const uint64_t base = kv_off[cursor];
  while (lo < hi) {
    uint32_t mid = lo + (hi - lo + 1) / 2;
    if (kv_off[cursor + mid] - base <= cap) lo = mid; else hi = mid - 1;
  }
  *out_count = lo;
}

struct KvIndexDev { uint32_t key_off, key_len, val_off, val_len, same_key; };

// one warp per record: copies key then value bytes into the batch buffer and fills the index entry
__global__ void __launch_bounds__(256)
    k_gather_batch(Records rec, const uint32_t *__restrict__ order, const uint8_t *__restrict__ same,
                   const uint64_t *__restrict__ kv_off, uint32_t cursor, uint32_t count, uint8_t *__restrict__ out,
                   KvIndexDev *__restrict__ idx, int check_same) {
  const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= count) return;
  const uint32_t r = cursor + w, i = order[r];
  const uint64_t o = kv_off[r] - kv_off[cursor];
  const uint32_t kl = rec.key_len[i], vl = rec.val_len[i];
  const uint8_t *k = rec.kv + rec.key_off[i];
  const uint8_t *v = rec.kv + (rec.val_off ? rec.val_off[i] : rec.key_off[i] + kl);
  for (uint32_t b = lane; b < kl; b += 32) out[o + b] = k[b];
  for (uint32_t b = lane; b < vl; b += 32) out[o + kl + b] = v[b];
  if (lane == 0) {
    KvIndexDev e;
    e.key_off = (uint32_t)o; e.key_len = kl; e.val_off = (uint32_t)(o + kl); e.val_len = vl;
    // MergeQueue.isSameKey(): read as SAME_KEY from its segment, or (checkForSameKeys) equal to the previous key of
    // another segment
    bool sk = false;
    if (r > 0 && same[r]) {
      const uint32_t tag = rec.tag[i], tagp = rec.tag[order[r - 1]];
      sk = (tag & 1u) || (check_same && ((tag >> 1) != (tagp >> 1)));
    }
    e.same_key = sk ? 1u : 0u;
    idx[w] = e;
  }
}

// ------------------------------------------------------------------------------------------------ host orchestration
class Merger {
 public:
  SortPipeline pipe;
  DeviceBuffer d_data, d_segs, d_piece_start, d_piece_crc, d_seg_crc, d_counts, d_rec_base;
  DeviceBuffer d_koff, d_voff, d_klen, d_vlen, d_tag, d_part, d_sizes, d_kvoff, d_batch, d_batch_idx, d_out;
  PinnedBuffer h_stage, h_out;
  std::vector<SegDesc> segs;
  uint64_t n = 0, kv_bytes = 0, seg_bytes = 0, cursor = 0;
  bool have_kvoff = false;
  int launches = 0;
  const uint8_t *data = nullptr;  // base of the segment bytes on the device

  static tezgpu_conf pipe_conf(tezgpu_conf c) {
    if (c.num_partitions < 1) c.num_partitions = 1;
    c.partitioner = TEZGPU_PART_GIVEN;
    if (c.num_partitions == 1) c.send_empty_partition_details = 0;  // a merge always writes its (possibly empty) segment
    c.fixed_key_len = c.fixed_val_len = 0;
    return c;
  }
  uint32_t fixed_klen = 0, fixed_vlen = 0;
  bool parsed_fixed = false;
  uint32_t data_slack = 32;

  explicit Merger(const tezgpu_conf &c) : pipe(pipe_conf(c)), fixed_klen(c.fixed_key_len), fixed_vlen(c.fixed_val_len) {}

  DeviceBuffer d_run_off, d_run_base, d_run_part, d_run_pseg, d_flags;
  std::vector<uint32_t> seg_orig;   // position in the partition-major list -> index in the caller's segment array
  bool arrays_ready = false;   // the per-record metadata arrays (d_koff ...) are filled (never in run-table mode unless asked)
  std::vector<uint64_t> h_counts, h_rec_base;

  void open(const tezgpu_segment *in, uint32_t nseg) {
    cudaStream_t st = pipe.stream;
    TG_CUDA(cudaSetDevice(pipe.conf.device));
    parsed_fixed = false;
    arrays_ready = false;
    // ---- segments already on this device are used in place (no copy; kernels handle any byte alignment);
    //      host segments are staged contiguously with 16-byte aligned starts
    segs.resize(nseg);
    bool all_device = nseg > 0;
    for (uint32_t s = 0; s < nseg; s++) all_device &= (in[s].flags & TEZGPU_SEG_DEVICE) != 0;
    uint64_t off = 0;
    uintptr_t lo_addr = ~(uintptr_t)0, hi_addr = 0;
    if (all_device)
      for (uint32_t s = 0; s < nseg; s++) {
        lo_addr = std::min(lo_addr, (uintptr_t)in[s].data);
        hi_addr = std::max(hi_addr, (uintptr_t)in[s].data + in[s].len);
      }
    lo_addr &= ~(uintptr_t)15;
    bool any_header = false;
    // Segments are kept partition-major (stable: the caller's order inside a partition is the merge's tie order): the
    // records of one output partition then live in a handful of consecutive runs, which makes the run-table lookups of
    // the stage / emit kernels a scan over <= G entries instead of a binary search over all segments.
    seg_orig.resize(nseg);
    for (uint32_t s = 0; s < nseg; s++) seg_orig[s] = s;
    if (pipe.conf.num_partitions > 1)
      std::stable_sort(seg_orig.begin(), seg_orig.end(), [&](uint32_t a, uint32_t b) { return in[a].partition < in[b].partition; });
    for (uint32_t s = 0; s < nseg; s++) {
      const tezgpu_segment &sg = in[seg_orig[s]];
      TG_CHECK(sg.data || sg.len == 0, TEZGPU_E_INVALID, "null segment");
      const bool hdr = sg.flags & TEZGPU_SEG_HAS_HEADER;
      any_header |= hdr;
      TG_CHECK(sg.len >= (hdr ? 10u : 6u), TEZGPU_E_FORMAT, "IFile segment shorter than an empty segment");
      segs[s].off = all_device ? (uint64_t)((uintptr_t)sg.data - lo_addr) : off;
      segs[s].len = sg.len;
      segs[s].body0 = hdr ? 4 : 0;
      segs[s].body_end = sg.len - 4;
      segs[s].has_header = (hdr ? 1u : 0u) | ((hdr && (sg.flags & TEZGPU_SEG_VERIFIED)) ? 2u : 0u);
      segs[s].partition = sg.partition;
      TG_CHECK((int)sg.partition < pipe.conf.num_partitions, TEZGPU_E_INVALID, "segment partition out of range");
      off = align_up(off + sg.len, 16);
    }
    if (all_device) {
      data = reinterpret_cast<const uint8_t *>(lo_addr);
      seg_bytes = (uint64_t)(hi_addr - lo_addr);
      data_slack = 0;  // caller's buffer: never read past its end
    } else {
      seg_bytes = off;
      d_data.ensure(off + 64);
      for (uint32_t s = 0; s < nseg; s++) {
        const tezgpu_segment &sg = in[seg_orig[s]];
        if (!sg.len) continue;
        const bool dev = sg.flags & TEZGPU_SEG_DEVICE;
        TG_CUDA(cudaMemcpyAsync(d_data.as<uint8_t>() + segs[s].off, sg.data, sg.len,
                                dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
      }
      data = d_data.as<uint8_t>();
      data_slack = 32;
    }
    d_segs.ensure((size_t)(nseg ? nseg : 1) * sizeof(SegDesc));
    if (nseg) TG_CUDA(cudaMemcpyAsync(d_segs.p, segs.data(), (size_t)nseg * sizeof(SegDesc), cudaMemcpyHostToDevice, st));
    // verdict words of the header / checksum checks: [0] bad magic, [1] compressed, [2] checksum mismatch (segment + 1).
    // They live outside the sorter's scratch so the whole fixed-framing path needs no host round trip before the sort.
    d_flags.ensure(64);
    TG_CUDA(cudaMemsetAsync(d_flags.p, 0, 64, st));
    int *d_vflags = d_flags.as<int>();
    const CrcTables *d_crc = DeviceConstants::get(pipe.conf.device).d_crc;
    if (nseg) {
      if (any_header) {
        k_check_headers<<<(uint32_t)div_up(nseg, 128), 128, 0, st>>>(data, d_segs.as<SegDesc>(), nseg, d_vflags, d_vflags + 1);
        launches++;
      }
      // ---- checksums of the segments nobody verified yet
      std::vector<uint32_t> piece_start(nseg + 1);
      uint32_t np = 0;
      for (uint32_t s = 0; s < nseg; s++) {
        piece_start[s] = np;
        if (segs[s].has_header == 1u) np += (uint32_t)div_up(segs[s].body_end - segs[s].body0, CRC_PIECE);
      }
      piece_start[nseg] = np;
      if (np) {
        d_piece_start.ensure((size_t)(nseg + 1) * 4);
        TG_CUDA(cudaMemcpyAsync(d_piece_start.p, piece_start.data(), (size_t)(nseg + 1) * 4, cudaMemcpyHostToDevice, st));
        TG_CUDA(cudaStreamSynchronize(st));  // piece_start is a stack-lifetime vector
        d_piece_crc.ensure((size_t)np * sizeof(TileCrc));
        d_seg_crc.ensure((size_t)nseg * 4);
        TG_CUDA(cudaMemsetAsync(d_seg_crc.p, 0, (size_t)nseg * 4, st));
        k_crc_pieces<<<np, CRCV_THREADS, 0, st>>>(data, d_segs.as<SegDesc>(), d_piece_start.as<uint32_t>(), nseg, d_crc,
                                                  d_piece_crc.as<TileCrc>());
        k_crc_combine<<<(uint32_t)div_up(np, 256), 256, 0, st>>>(d_piece_crc.as<TileCrc>(), np, d_crc, d_seg_crc.as<uint32_t>());
        k_crc_check<<<(uint32_t)div_up(nseg, 128), 128, 0, st>>>(data, d_segs.as<SegDesc>(), nseg, d_seg_crc.as<uint32_t>(), d_crc, d_vflags + 2);
        launches += 3;
        TG_CUDA(cudaGetLastError());
      }
    }
    auto check_verdicts = [&]() {
      int f[3] = {0, 0, 0};
      TG_CUDA(cudaMemcpyAsync(f, d_vflags, 12, cudaMemcpyDeviceToHost, st));
      TG_CUDA(cudaStreamSynchronize(st));
      TG_CHECK(f[0] == 0, TEZGPU_E_FORMAT, "Not a valid ifile header (segment " + std::to_string(f[0] ? seg_orig[f[0] - 1] : 0) + ")");
      TG_CHECK(f[1] == 0, TEZGPU_E_UNSUPPORTED, "compressed IFile segments are not supported on the device path");
      TG_CHECK(f[2] == 0, TEZGPU_E_FORMAT, "IFile checksum mismatch in segment " + std::to_string(f[2] ? seg_orig[f[2] - 1] : 0));
    };

    // ---- records per segment
    h_counts.assign(2 * (size_t)nseg + 2, 0);
    h_rec_base.assign(nseg + 1, 0);
    bool fixed_ok = false;
    const uint32_t rs = vint_size_u32(fixed_klen) + vint_size_u32(fixed_vlen) + fixed_klen + fixed_vlen;
    if (nseg && fixed_klen + fixed_vlen > 0) {
      // candidate: every body is exactly k records of the fixed framing + EOF markers
      fixed_ok = true;
      for (uint32_t s = 0; s < nseg && fixed_ok; s++) {
        uint64_t body = segs[s].body_end - segs[s].body0;
        fixed_ok = body >= 2 && (body - 2) % rs == 0;
        h_counts[s] = fixed_ok ? (body - 2) / rs : 0;
        h_counts[nseg + s] = h_counts[s] * (fixed_klen + fixed_vlen);
      }
    }
    if (fixed_ok) {
      // ---- run-table mode: offsets are arithmetic, the stage kernel checks the framing bytes it passes over anyway.
      //      No per-record arrays, no host round trip before the sort's own.
      n = 0;
      kv_bytes = 0;
      for (uint32_t s = 0; s < nseg; s++) { h_rec_base[s] = n; n += h_counts[s]; kv_bytes += h_counts[nseg + s]; }
      h_rec_base[nseg] = n;
      TG_CHECK(n <= RADIX_MAX_N, TEZGPU_E_INVALID, "more than 2^30-1 records in one merge");
      std::vector<uint64_t> roff(nseg);
      std::vector<uint32_t> rbase(nseg + 1), rpart(nseg);
      for (uint32_t s = 0; s < nseg; s++) { roff[s] = segs[s].off + segs[s].body0; rbase[s] = (uint32_t)h_rec_base[s]; rpart[s] = segs[s].partition; }
      rbase[nseg] = (uint32_t)n;
      const int P = pipe.conf.num_partitions;
      std::vector<uint32_t> pseg((size_t)P + 1, 0);
      for (uint32_t s = 0; s < nseg; s++) pseg[segs[s].partition + 1]++;
      uint32_t max_runs = 0;
      for (int p = 0; p < P; p++) { max_runs = std::max(max_runs, pseg[p + 1]); pseg[p + 1] += pseg[p]; }
      pipe.merge_max_runs = max_runs;
      d_run_pseg.ensure(((size_t)P + 1) * 4);
      TG_CUDA(cudaMemcpyAsync(d_run_pseg.p, pseg.data(), ((size_t)P + 1) * 4, cudaMemcpyHostToDevice, st));
      d_run_off.ensure((size_t)nseg * 8); d_run_base.ensure((size_t)(nseg + 1) * 4); d_run_part.ensure((size_t)nseg * 4);
      TG_CUDA(cudaMemcpyAsync(d_run_off.p, roff.data(), (size_t)nseg * 8, cudaMemcpyHostToDevice, st));
      TG_CUDA(cudaMemcpyAsync(d_run_base.p, rbase.data(), (size_t)(nseg + 1) * 4, cudaMemcpyHostToDevice, st));
      TG_CUDA(cudaMemcpyAsync(d_run_part.p, rpart.data(), (size_t)nseg * 4, cudaMemcpyHostToDevice, st));
      TG_CUDA(cudaStreamSynchronize(st));  // stack-lifetime staging vectors (and: the caller's host segments may go away)
      Records r;
      memset(&r, 0, sizeof(r));
      r.kv = data;
      r.kv_bytes = data_slack ? align_up(seg_bytes, 16) + data_slack : seg_bytes;
      r.n = (uint32_t)n;
      r.fixed = 1;
      r.klen = fixed_klen;
      r.vlen = fixed_vlen;
      r.use_runs = 1;
      r.runs.seg_off = d_run_off.as<uint64_t>();
      r.runs.rec_base = d_run_base.as<uint32_t>();
      r.runs.seg_part = d_run_part.as<uint32_t>();
      r.runs.part_seg0 = d_run_pseg.as<uint32_t>();
      r.runs.nseg = nseg;
      r.runs.rec_size = rs;
      r.runs.hdr_len = vint_size_u32(fixed_klen) + vint_size_u32(fixed_vlen);
      uint64_t hb = 0;
      int b = 0;
      for (int i = 0; i < vint_size_u32(fixed_klen); i++) hb |= (uint64_t)vint_byte_u32(fixed_klen, i) << (8 * b++);
      for (int i = 0; i < vint_size_u32(fixed_vlen); i++) hb |= (uint64_t)vint_byte_u32(fixed_vlen, i) << (8 * b++);
      r.runs.hdr_bytes = hb;
      bool mismatch = false;
      pipe.merge_inputs_plain = true;
      try {
        pipe.sort_phase(r);
      } catch (const FramingMismatch &) {
        mismatch = true;  // not the fixed framing after all (e.g. run-length encoded input): take the general walk
      }
      check_verdicts();
      if (!mismatch) {
        parsed_fixed = true;
        parse_mode = 0;
        parse_rounds = 0;
        launches += pipe.state.launches;
        cursor = 0;
        have_kvoff = false;
        return;
      }
    } else {
      check_verdicts();  // also: the caller's host buffers may go away after open()
    }

    // ---- general path: walk the segments (IFile.Reader semantics), materialise the per-record metadata
    int *d_bad = pipe.d_error();
    TG_CUDA(cudaMemsetAsync(pipe.small.p, 0, 16384, st));
    d_counts.ensure((size_t)(nseg + 1) * 16);
    d_rec_base.ensure((size_t)(nseg + 2) * 8);
    n = 0;
    kv_bytes = 0;
    if (nseg) open_general_reparse(nseg, h_counts, h_rec_base);
    else {
      d_koff.ensure(8); d_voff.ensure(8); d_klen.ensure(4); d_vlen.ensure(4); d_tag.ensure(4); d_part.ensure(4);
    }
    (void)d_bad;
    TG_CUDA(cudaGetLastError());
    arrays_ready = true;

    // ---- merge = stable sort of the union of the runs by the RawComparator
    Records r = array_records();
    pipe.merge_inputs_plain = false;
    pipe.sort_phase(r);
    launches += pipe.state.launches;
    cursor = 0;
    have_kvoff = false;
  }

  // Records over the materialised per-record arrays
  Records array_records() {
    Records r;
    memset(&r, 0, sizeof(r));
    r.kv = data;
    r.kv_bytes = data_slack ? align_up(seg_bytes, 16) + data_slack : seg_bytes;
    r.key_off = d_koff.as<uint64_t>();
    r.val_off = d_voff.as<uint64_t>();
    r.key_len = d_klen.as<uint32_t>();
    r.val_len = d_vlen.as<uint32_t>();
    r.tag = d_tag.as<uint32_t>();
    r.partition = pipe.conf.num_partitions > 1 ? d_part.as<int32_t>() : nullptr;
    r.n = (uint32_t)n;
    r.fixed = 0;
    return r;
  }

  // run-table mode keeps no per-record arrays; the record iterator and the general (run-length encoding) emit need
  // them: fill them now (same record numbering, so the sorted order stays valid) and switch the sorter's view over
  void ensure_arrays() {
    if (arrays_ready) return;
    cudaStream_t st = pipe.stream;
    const uint32_t nseg = (uint32_t)segs.size();
    d_rec_base.ensure((size_t)(nseg + 2) * 8);
    TG_CUDA(cudaMemcpyAsync(d_rec_base.p, h_rec_base.data(), (size_t)(nseg + 1) * 8, cudaMemcpyHostToDevice, st));
    d_koff.ensure((size_t)(n ? n : 1) * 8); d_voff.ensure((size_t)(n ? n : 1) * 8);
    d_klen.ensure((size_t)(n ? n : 1) * 4); d_vlen.ensure((size_t)(n ? n : 1) * 4); d_tag.ensure((size_t)(n ? n : 1) * 4); d_part.ensure((size_t)(n ? n : 1) * 4);
    ParseArrays pa{d_koff.as<uint64_t>(), d_voff.as<uint64_t>(), d_klen.as<uint32_t>(), d_vlen.as<uint32_t>(), d_tag.as<uint32_t>(), d_part.as<int32_t>()};
    if (n) {
      const uint32_t hl = vint_size_u32(fixed_klen) + vint_size_u32(fixed_vlen);
      k_fill_fixed_arrays<<<(uint32_t)std::min<uint64_t>(div_up(n, 256), 148 * 16), 256, 0, st>>>(
          d_segs.as<SegDesc>(), nseg, d_rec_base.as<uint64_t>(), fixed_klen, fixed_vlen, hl, pa);
      launches++;
      TG_CUDA(cudaGetLastError());
    }
    Records r = array_records();
    r.fixed = 1;
    r.klen = fixed_klen;
    r.vlen = fixed_vlen;
    r.cmp = pipe.state.rec.cmp;
    r.hash_partition = pipe.state.rec.hash_partition;
    r.num_partitions = pipe.state.rec.num_partitions;
    r.pbits = pipe.state.rec.pbits;
    pipe.state.rec = r;
    // the record view changed (explicit offsets instead of the run table): the emit must lay its tiles out again --
    // tile sizes depend on the kernel that serves the view (set_fixed_layout)
    pipe.state.spec_layout = false;
    arrays_ready = true;
  }

  // ---- parallel parser (parse_windows.cuh): every window of every segment walks at once, entries iterate to the fixed
  // point.  Returns false when the rounds cap is hit (adversarial bytes): the caller falls back to the sequential walker.
  DeviceBuffer d_pwseg, d_entry[2], d_wcount, d_wbase, d_wlast, d_carry, d_pwflags;
  int parse_rounds = 0;
  int parse_mode = 0;   // how the last open() found the records: 0 fixed framing (run table), 1 window parser, 2 sequential walker
  bool parse_parallel(uint32_t nseg) {
    cudaStream_t st = pipe.stream;
    std::vector<PwSeg> ps(nseg);
    uint64_t nw = 0;
    for (uint32_t s = 0; s < nseg; s++) {
      ps[s].off = segs[s].off; ps[s].len = segs[s].len; ps[s].body0 = segs[s].body0; ps[s].body_end = segs[s].body_end;
      ps[s].win0 = (uint32_t)nw;
      ps[s].nwin = (uint32_t)std::max<uint64_t>(1, div_up(segs[s].body_end - segs[s].body0, PW_WINDOW));
      ps[s].partition = segs[s].partition;
      ps[s].pad = 0;
      nw += ps[s].nwin;
    }
    TG_CHECK(nw < (1ull << 31), TEZGPU_E_INVALID, "segments too large for one merge");
    const uint32_t nwin = (uint32_t)nw;
    d_pwseg.ensure((size_t)nseg * sizeof(PwSeg));
    for (int b = 0; b < 2; b++) d_entry[b].ensure((size_t)nwin * 8);
    d_wcount.ensure((size_t)nwin * 4);
    d_wbase.ensure(((size_t)nwin + 2) * 8);
    d_wlast.ensure((size_t)nwin * 16);
    d_pwflags.ensure(64);
    TG_CUDA(cudaMemcpyAsync(d_pwseg.p, ps.data(), (size_t)nseg * sizeof(PwSeg), cudaMemcpyHostToDevice, st));
    const uint32_t grid = (uint32_t)div_up(nwin, PW_THREADS);
    PwArrays none{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // guess -> evaluate from the guessed entries -> chase the true chain (parse_windows.cuh); one host round trip
    TG_CUDA(cudaMemsetAsync(d_pwflags.p, 0, 64, st));
    PwFixedHint hint{0, 0, 0, 0};
    if (fixed_klen + fixed_vlen > 0 && vint_size_u32(fixed_klen) + vint_size_u32(fixed_vlen) <= 7) {
      int b = 0;
      for (int i = 0; i < vint_size_u32(fixed_klen); i++) hint.full |= (uint64_t)vint_byte_u32(fixed_klen, i) << (8 * b++);
      for (int i = 0; i < vint_size_u32(fixed_vlen); i++) hint.full |= (uint64_t)vint_byte_u32(fixed_vlen, i) << (8 * b++);
      hint.full_len = (uint32_t)b;
      for (int i = 0; i < vint_size_u32(fixed_vlen); i++) hint.rep |= (uint64_t)vint_byte_u32(fixed_vlen, i) << (8 * i);
      hint.rep_len = (uint32_t)vint_size_u32(fixed_vlen);
    }
    k_parse_guess<<<(uint32_t)div_up((uint64_t)nwin * 32, PW_GUESS_THREADS), PW_GUESS_THREADS, 0, st>>>(data, d_pwseg.as<PwSeg>(), nseg, nwin,
                                                                                                        d_entry[0].as<uint64_t>(), hint);
    k_parse_windows<1><<<grid, PW_THREADS, 0, st>>>(data, d_pwseg.as<PwSeg>(), nseg, nwin, d_entry[0].as<uint64_t>(),
                                                    d_entry[1].as<uint64_t>(), d_wcount.as<uint32_t>(), d_wlast.as<uint64_t>(),
                                                    nullptr, d_pwflags.as<int>(), nullptr, nullptr, none);
    k_parse_chase<<<(uint32_t)div_up(nseg, PW_CHASE_WARPS), 32 * PW_CHASE_WARPS, 0, st>>>(
        data, d_pwseg.as<PwSeg>(), nseg, d_entry[0].as<uint64_t>(), d_entry[1].as<uint64_t>(), d_wcount.as<uint32_t>(),
        d_wlast.as<uint64_t>(), d_pwflags.as<int>());
    launches += 3;
    TG_CUDA(cudaGetLastError());
    int flags[4] = {0, 0, 0, 0};
    TG_CUDA(cudaMemcpyAsync(flags, d_pwflags.p, 16, cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaStreamSynchronize(st));
    parse_rounds = flags[2];   // windows the chase had to walk by hand
    // the sequential reader would reject a segment (or it ends early): the sequential walker reports it
    if (flags[1]) return false;
    const int cur = 0;         // d_entry[0] now holds the true entries
    // ---- record offsets of every window, totals
    const uint32_t nblk = (uint32_t)div_up(nwin, SCAN_TILE);
    pipe.blk.ensure(((size_t)nblk + 2) * 8);
    k_sum_u32_blocks<<<nblk, SCAN_THREADS, 0, st>>>(d_wcount.as<uint32_t>(), nwin, pipe.blk.as<uint64_t>());
    k_scan_block_sums<<<1, 1024, 0, st>>>(pipe.blk.as<uint64_t>(), nblk);
    k_scan_u32_apply<<<nblk, SCAN_THREADS, 0, st>>>(d_wcount.as<uint32_t>(), nwin, pipe.blk.as<uint64_t>(), d_wbase.as<uint64_t>());
    d_counts.ensure((size_t)(nseg + 1) * 16);
    k_parse_seg_counts<<<(uint32_t)div_up(nseg, 128), 128, 0, st>>>(d_pwseg.as<PwSeg>(), nseg, d_wbase.as<uint64_t>(), d_counts.as<uint64_t>());
    launches += 4;
    uint64_t total = 0;
    TG_CUDA(cudaMemcpyAsync(&total, d_wbase.as<uint64_t>() + nwin, 8, cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaMemcpyAsync(h_counts.data(), d_counts.p, (size_t)nseg * 8, cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaStreamSynchronize(st));
    n = total;
    TG_CHECK(n <= RADIX_MAX_N, TEZGPU_E_INVALID, "more than 2^30-1 records in one merge");
    uint64_t acc = 0;
    for (uint32_t s = 0; s < nseg; s++) { h_rec_base[s] = acc; acc += h_counts[s]; }
    h_rec_base[nseg] = acc;
    d_koff.ensure((size_t)(n ? n : 1) * 8); d_voff.ensure((size_t)(n ? n : 1) * 8);
    d_klen.ensure((size_t)(n ? n : 1) * 4); d_vlen.ensure((size_t)(n ? n : 1) * 4); d_tag.ensure((size_t)(n ? n : 1) * 4); d_part.ensure((size_t)(n ? n : 1) * 4);
    PwArrays pa{d_koff.as<uint64_t>(), d_voff.as<uint64_t>(), d_klen.as<uint32_t>(), d_vlen.as<uint32_t>(), d_tag.as<uint32_t>(), d_part.as<int32_t>()};
    d_carry.ensure((size_t)nwin * 16);
    k_parse_carry<<<grid, PW_THREADS, 0, st>>>(d_pwseg.as<PwSeg>(), nseg, nwin, d_entry[cur].as<uint64_t>(), d_wlast.as<uint64_t>(), d_carry.as<uint64_t>());
    const uint64_t *carry = d_carry.as<uint64_t>();
    launches++;
    TG_CUDA(cudaMemsetAsync(d_pwflags.p, 0, 64, st));
    unsigned long long *d_kv_total = reinterpret_cast<unsigned long long *>(d_pwflags.as<int>() + 8);
    k_parse_windows<2><<<(uint32_t)div_up((uint64_t)nwin * PW_EMIT_GROUP, PW_THREADS), PW_THREADS, 0, st>>>(data, d_pwseg.as<PwSeg>(), nseg, nwin, d_entry[cur].as<uint64_t>(), nullptr, nullptr, nullptr,
                                                       d_kv_total, d_pwflags.as<int>(), d_wbase.as<uint64_t>(), carry, pa);
    launches++;
    TG_CUDA(cudaGetLastError());
    unsigned long long kvb = 0;
    TG_CUDA(cudaMemcpyAsync(flags, d_pwflags.p, 16, cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaMemcpyAsync(&kvb, d_kv_total, 8, cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaStreamSynchronize(st));
    TG_CHECK(flags[1] == 0, TEZGPU_E_FORMAT, "malformed IFile segment " + std::to_string(flags[1] ? seg_orig[flags[1] - 1] : 0));
    kv_bytes = kvb;
    return true;
  }

  void open_general_reparse(uint32_t nseg, std::vector<uint64_t> &counts, std::vector<uint64_t> &rec_base) {
    cudaStream_t st = pipe.stream;
    static const bool serial_only = getenv("TEZGPU_PARSE_SERIAL") && atoi(getenv("TEZGPU_PARSE_SERIAL")) != 0;
    parse_mode = 1;
    if (!serial_only && parse_parallel(nseg)) return;
    parse_mode = 2;
    int *d_bad = pipe.d_error();
    ParseArrays pa{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    k_parse_segments<false><<<(uint32_t)div_up(nseg, PARSE_WARPS), PARSE_WARPS * 32, 0, st>>>(data, d_segs.as<SegDesc>(), nseg, d_counts.as<uint64_t>(),
                                                                     d_counts.as<uint64_t>() + nseg, nullptr, pa, d_bad);
    int bad = 0;
    TG_CUDA(cudaMemcpyAsync(counts.data(), d_counts.p, (size_t)nseg * 16, cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaStreamSynchronize(st));
    TG_CHECK(bad == 0, TEZGPU_E_FORMAT, "malformed IFile segment " + std::to_string(bad ? seg_orig[bad - 1] : 0));
    n = 0;
    kv_bytes = 0;
    for (uint32_t s = 0; s < nseg; s++) { rec_base[s] = n; n += counts[s]; kv_bytes += counts[nseg + s]; }
    rec_base[nseg] = n;
    TG_CHECK(n <= RADIX_MAX_N, TEZGPU_E_INVALID, "more than 2^30-1 records in one merge");
    TG_CUDA(cudaMemcpyAsync(d_rec_base.p, rec_base.data(), (size_t)(nseg + 1) * 8, cudaMemcpyHostToDevice, st));
    d_koff.ensure((size_t)(n ? n : 1) * 8); d_voff.ensure((size_t)(n ? n : 1) * 8);
    d_klen.ensure((size_t)(n ? n : 1) * 4); d_vlen.ensure((size_t)(n ? n : 1) * 4); d_tag.ensure((size_t)(n ? n : 1) * 4); d_part.ensure((size_t)(n ? n : 1) * 4);
    pa = ParseArrays{d_koff.as<uint64_t>(), d_voff.as<uint64_t>(), d_klen.as<uint32_t>(), d_vlen.as<uint32_t>(), d_tag.as<uint32_t>(), d_part.as<int32_t>()};
    if (n) k_parse_segments<true><<<(uint32_t)div_up(nseg, PARSE_WARPS), PARSE_WARPS * 32, 0, st>>>(data, d_segs.as<SegDesc>(), nseg, nullptr, nullptr,
                                                                            d_rec_base.as<uint64_t>(), pa, d_bad);
    launches += 2;
  }

  uint64_t output_bound() const { return SortPipeline::output_bound(n, kv_bytes, pipe.conf.num_partitions) + 16; }

  // TezMerger.writeFile: one IFile segment, equal adjacent keys written through IFile.REPEAT_KEY
  void write_device(uint8_t *d_out_buf, uint64_t cap, int writer_rle, int64_t *raw_len, int64_t *part_len, tezgpu_stats *stats) {
    TG_CHECK(pipe.conf.num_partitions == 1, TEZGPU_E_STATE,
             "merger was opened with num_partitions > 1: use tezgpu_merge_write_partitions*");
    int64_t index[3] = {0, 0, 0};
    uint64_t len = 0;
    tezgpu_stats st;
    pipe.emit_output(writer_rle ? 1 : 0, true, d_out_buf, cap, &len, index, &st);
    st.output_bytes = (int64_t)kv_bytes;
    st.kernel_launches += launches - pipe.state.launches;
    if (raw_len) *raw_len = index[1];
    if (part_len) *part_len = index[2];
    if (stats) *stats = st;
  }

  void write_partitions_device(uint8_t *d_out_buf, uint64_t cap, int writer_rle, uint64_t *out_len, int64_t *index,
                               tezgpu_stats *stats) {
    tezgpu_stats st;
    pipe.emit_output(writer_rle ? 1 : 0, true, d_out_buf, cap, out_len, index, &st);
    st.output_bytes = (int64_t)kv_bytes;
    st.kernel_launches += launches - pipe.state.launches;
    if (stats) *stats = st;
  }

  void ensure_kvoff() {
    if (have_kvoff) return;
    ensure_arrays();
    cudaStream_t st = pipe.stream;
    const uint32_t nn = (uint32_t)n;
    d_sizes.ensure((size_t)(nn ? nn : 1) * 4);
    d_kvoff.ensure(((size_t)nn + 2) * 8);
    if (nn) {
      const uint32_t nblk = (uint32_t)div_up(nn, SCAN_TILE);
      pipe.blk.ensure(((size_t)nblk + 2) * 8);
      k_kv_sizes<<<(uint32_t)div_up(nn, 256), 256, 0, st>>>(pipe.state.rec, pipe.state.order, d_sizes.as<uint32_t>());
      k_sum_u32_blocks<<<nblk, SCAN_THREADS, 0, st>>>(d_sizes.as<uint32_t>(), nn, pipe.blk.as<uint64_t>());
      k_scan_block_sums<<<1, 1024, 0, st>>>(pipe.blk.as<uint64_t>(), nblk);
      k_scan_u32_apply<<<nblk, SCAN_THREADS, 0, st>>>(d_sizes.as<uint32_t>(), nn, pipe.blk.as<uint64_t>(), d_kvoff.as<uint64_t>());
      TG_CUDA(cudaGetLastError());
    } else {
      TG_CUDA(cudaMemsetAsync(d_kvoff.p, 0, 16, st));
    }
    have_kvoff = true;
  }

  // next()/getKey()/getValue()/isSameKey() in batches
  void next_batch(uint8_t *out_kv, uint64_t cap, tezgpu_kv_index *idx, uint32_t idx_cap, uint32_t *count) {
    TG_CUDA(cudaSetDevice(pipe.conf.device));
    cudaStream_t st = pipe.stream;
    *count = 0;
    if (cursor >= n || idx_cap == 0) return;
    ensure_kvoff();
    uint32_t *d_cnt = pipe.d_large();
    k_find_batch<<<1, 1, 0, st>>>(d_kvoff.as<uint64_t>(), (uint32_t)n, (uint32_t)cursor, idx_cap, cap, d_cnt);
    uint32_t cnt = 0;
    TG_CUDA(cudaMemcpyAsync(&cnt, d_cnt, 4, cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaStreamSynchronize(st));
    TG_CHECK(cnt > 0, TEZGPU_E_NOMEM, "batch buffer smaller than one record");
    uint64_t ends[2];
    TG_CUDA(cudaMemcpyAsync(&ends[0], d_kvoff.as<uint64_t>() + cursor, 8, cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaMemcpyAsync(&ends[1], d_kvoff.as<uint64_t>() + cursor + cnt, 8, cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaStreamSynchronize(st));
    const uint64_t bytes = ends[1] - ends[0];
    d_batch.ensure(bytes + 16);
    d_batch_idx.ensure((size_t)cnt * sizeof(KvIndexDev));
    k_gather_batch<<<(uint32_t)div_up((uint64_t)cnt * 32, 256), 256, 0, st>>>(pipe.state.rec, pipe.state.order, pipe.same.as<uint8_t>(),
                                                                         d_kvoff.as<uint64_t>(), (uint32_t)cursor, cnt,
                                                                         d_batch.as<uint8_t>(), d_batch_idx.as<KvIndexDev>(),
                                                                         pipe.merge_check_same);
    TG_CUDA(cudaGetLastError());
    if (bytes) TG_CUDA(cudaMemcpyAsync(out_kv, d_batch.p, bytes, cudaMemcpyDeviceToHost, st));
    static_assert(sizeof(KvIndexDev) == sizeof(tezgpu_kv_index), "index layout");
    TG_CUDA(cudaMemcpyAsync(idx, d_batch_idx.p, (size_t)cnt * sizeof(KvIndexDev), cudaMemcpyDeviceToHost, st));
    TG_CUDA(cudaStreamSynchronize(st));
    cursor += cnt;
    *count = cnt;
  }
};

}  // namespace tezgpu
