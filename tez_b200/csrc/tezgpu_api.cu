// tezgpu_api.cu -- extern "C" boundary of libtezgpu.so (include/tezgpu.h).  No CPU fallback: every compute entry
// point needs a CUDA device and fails with TEZGPU_E_CUDA otherwise.
#include <errno.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <mutex>
#include <string>

#include "../../include/tezgpu.h"
#include "merger.cuh"
#include "sorter.cuh"
#include "peer_fetch.cuh"

using namespace tezgpu;

static thread_local std::string g_last_error;

#define TG_API_BEGIN try {
#define TG_API_END                                  \
  }                                                 \
  catch (const tezgpu::Error &e) {                  \
    g_last_error = e.what();                        \
    return e.code;                                  \
  }                                                 \
  catch (const std::bad_alloc &) {                  \
    g_last_error = "host allocation failed";        \
    return TEZGPU_E_NOMEM;                          \
  }                                                 \
  catch (const std::exception &e) {                 \
    g_last_error = e.what();                        \
    return TEZGPU_E_INVALID;                        \
  }                                                 \
  return TEZGPU_OK;

// TezSpillRecord.writeToFile layout (SORT/TezSpillRecord.java:111-146): P x 3 big-endian longs + CRC32 as a long
static void spill_record_bytes(const int64_t *idx, int P, std::vector<uint8_t> &out) {
  out.resize((size_t)P * 24 + 8);
  for (int i = 0; i < P * 3; i++)
    for (int b = 0; b < 8; b++) out[(size_t)i * 8 + b] = (uint8_t)((uint64_t)idx[i] >> (56 - 8 * b));
  CrcTables *t = new CrcTables();
  crc_build_tables(*t, 1);
  uint32_t c = 0xFFFFFFFFu;
  for (size_t i = 0; i < (size_t)P * 24; i++) c = t->slice[0][(c ^ out[i]) & 0xFF] ^ (c >> 8);
  c = ~c;
  delete t;
  for (int b = 0; b < 8; b++) out[(size_t)P * 24 + b] = (uint8_t)((uint64_t)c >> (56 - 8 * b));
}

static void write_file_0640(const char *path, const void *data, size_t len) {
  // SPILL_FILE_PERMS = 0640 (SORT/TezSpillRecord.java:41,148-152)
  int fd = ::open(path, O_WRONLY | O_CREAT | O_TRUNC, 0640);
  TG_CHECK(fd >= 0, TEZGPU_E_IO, std::string("open ") + path + ": " + strerror(errno));
  const uint8_t *p = (const uint8_t *)data;
  size_t left = len;
  while (left) {
    ssize_t w = ::write(fd, p, left);
    if (w < 0) {
      if (errno == EINTR) continue;
      int e = errno;
      ::close(fd);
      throw Error(TEZGPU_E_IO, std::string("write ") + path + ": " + strerror(e));
    }
    p += w;
    left -= (size_t)w;
  }
  ::fchmod(fd, 0640);
  TG_CHECK(::close(fd) == 0, TEZGPU_E_IO, std::string("close ") + path + ": " + strerror(errno));
}

struct tezgpu_sorter {
  SortPipeline pipe;
  bool fixed;
  uint32_t klen, vlen;
  uint64_t n = 0, kv_bytes = 0, payload_bytes = 0;
  bool has_partition = false;
  bool flushed = false;
  DeviceBuffer d_kv, d_koff, d_klen, d_vlen, d_part, d_tmp, d_out;
  PinnedBuffer h_out;
  explicit tezgpu_sorter(const tezgpu_conf &c) : pipe(c) {
    fixed = c.fixed_key_len > 0 || c.fixed_val_len > 0;
    klen = c.fixed_key_len;
    vlen = c.fixed_val_len;
  }
  Records records() {
    Records r;
    memset(&r, 0, sizeof(r));
    r.kv = d_kv.as<uint8_t>();
    r.kv_bytes = align_up(kv_bytes, 16);
    r.key_off = d_koff.as<uint64_t>();
    r.key_len = d_klen.as<uint32_t>();
    r.val_len = d_vlen.as<uint32_t>();
    r.partition = has_partition ? d_part.as<int32_t>() : nullptr;
    r.n = (uint32_t)n;
    r.klen = klen;
    r.vlen = vlen;
    r.fixed = fixed;
    return r;
  }
};

__global__ void k_rebase_offsets(const uint32_t *__restrict__ key_off, const uint32_t *__restrict__ val_off,
                                 const uint32_t *__restrict__ val_len, uint32_t n, uint64_t base, uint64_t kv_bytes,
                                 uint64_t *__restrict__ koff64, uint32_t *__restrict__ klen, uint32_t *__restrict__ vlen,
                                 int *__restrict__ err) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t ko = key_off[i], vo = val_off[i], vl = val_len[i];
  if (vo < ko || (uint64_t)vo + vl > kv_bytes) { *err = 1; vo = ko; vl = 0; }
  koff64[i] = base + ko;
  klen[i] = vo - ko;
  vlen[i] = vl;
}

extern "C" {

const char *tezgpu_last_error(void) { return g_last_error.c_str(); }
int32_t tezgpu_abi_version(void) { return TEZGPU_ABI_VERSION; }
int32_t tezgpu_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int32_t tezgpu_sorter_create(const tezgpu_conf *conf, tezgpu_sorter **out) {
  TG_API_BEGIN
  TG_CHECK(conf && out, TEZGPU_E_INVALID, "null argument");
  TG_CHECK(conf->abi_version == TEZGPU_ABI_VERSION, TEZGPU_E_INVALID, "tezgpu_conf.abi_version mismatch");
  *out = new tezgpu_sorter(*conf);
  TG_API_END
}

int32_t tezgpu_sorter_destroy(tezgpu_sorter *h) {
  TG_API_BEGIN
  delete h;
  TG_API_END
}

int32_t tezgpu_sorter_reset(tezgpu_sorter *h) {
  TG_API_BEGIN
  TG_CHECK(h, TEZGPU_E_INVALID, "null handle");
  h->n = h->kv_bytes = h->payload_bytes = 0;
  h->has_partition = false;
  h->flushed = false;
  TG_API_END
}

int32_t tezgpu_sorter_collect_batch(tezgpu_sorter *h, const uint8_t *kv, uint64_t kv_bytes, const uint32_t *key_off,
                                    const uint32_t *val_off, const uint32_t *val_len, const int32_t *partition,
                                    uint32_t n) {
  TG_API_BEGIN
  TG_CHECK(h, TEZGPU_E_INVALID, "null handle");
  TG_CHECK(!h->flushed, TEZGPU_E_STATE, "collect after flush");
  TG_CHECK(!h->fixed, TEZGPU_E_STATE, "handle is in fixed-width mode: use tezgpu_sorter_collect_fixed");
  if (n == 0) return TEZGPU_OK;
  TG_CHECK(kv && key_off && val_off && val_len, TEZGPU_E_INVALID, "null argument");
  TG_CHECK(kv_bytes < (1ull << 32), TEZGPU_E_INVALID, "batch larger than 4 GiB");
  TG_CHECK(h->n + n <= RADIX_MAX_N, TEZGPU_E_INVALID, "more than 2^30-1 records collected");
  TG_CHECK((h->n == 0) || (h->has_partition == (partition != nullptr)), TEZGPU_E_INVALID,
           "partition ids must be given for all batches or none");
  TG_CHECK(partition || h->pipe.conf.partitioner == TEZGPU_PART_HASH, TEZGPU_E_INVALID,
           "partition ids required (partitioner=GIVEN)");
  {
    // the sort memory granted to this output (ExternalSorter.getInitialMemoryRequirement, SORT/ExternalSorter.java:330-347;
    // PipelinedSorter spills when its kvbuffer is full, :415-444): past it the caller must spill -- flush + reset --
    // first.  A first batch larger than the whole budget is still taken (the reference writes such records through).
    uint64_t add = 0;
    for (uint32_t i = 0; i < n; i++) add += (uint64_t)(val_off[i] - key_off[i]) + val_len[i];
    const uint64_t budget = h->pipe.conf.mem_budget_bytes;
    TG_CHECK(budget == 0 || h->n == 0 || h->payload_bytes + add <= budget, TEZGPU_E_NOMEM,
             "sort memory budget exceeded (" + std::to_string(h->payload_bytes + add) + " > " + std::to_string(budget) +
                 " bytes): spill (flush + reset) before collecting more");
  }
  cudaStream_t st = h->pipe.stream;
  TG_CUDA(cudaSetDevice(h->pipe.conf.device));
  const uint64_t base = align_up(h->kv_bytes, 16);  // every batch starts 16-byte aligned
  h->d_kv.grow_preserve(base + kv_bytes + 32, h->kv_bytes, st);
  h->d_koff.grow_preserve((h->n + n) * 8, h->n * 8, st);
  h->d_klen.grow_preserve((h->n + n) * 4, h->n * 4, st);
  h->d_vlen.grow_preserve((h->n + n) * 4, h->n * 4, st);
  if (partition) h->d_part.grow_preserve((h->n + n) * 4, h->n * 4, st);
  h->d_tmp.ensure((size_t)n * 12);
  uint32_t *t = h->d_tmp.as<uint32_t>();
  TG_CUDA(cudaMemcpyAsync(h->d_kv.as<uint8_t>() + base, kv, kv_bytes, cudaMemcpyHostToDevice, st));
  TG_CUDA(cudaMemcpyAsync(t, key_off, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  TG_CUDA(cudaMemcpyAsync(t + n, val_off, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  TG_CUDA(cudaMemcpyAsync(t + 2 * (size_t)n, val_len, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  if (partition)
    TG_CUDA(cudaMemcpyAsync(h->d_part.as<int32_t>() + h->n, partition, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  TG_CUDA(cudaMemsetAsync(h->pipe.d_error(), 0, 4, st));
  k_rebase_offsets<<<(uint32_t)div_up(n, 256), 256, 0, st>>>(t, t + n, t + 2 * (size_t)n, n, base, kv_bytes,
                                                           h->d_koff.as<uint64_t>() + h->n, h->d_klen.as<uint32_t>() + h->n,
                                                           h->d_vlen.as<uint32_t>() + h->n, h->pipe.d_error());
  TG_CUDA(cudaGetLastError());
  int err = 0;
  TG_CUDA(cudaMemcpyAsync(&err, h->pipe.d_error(), 4, cudaMemcpyDeviceToHost, st));
  TG_CUDA(cudaStreamSynchronize(st));  // caller may reuse its buffers once we return
  TG_CHECK(err == 0, TEZGPU_E_INVALID, "record offsets outside the batch buffer");
  for (uint32_t i = 0; i < n; i++) h->payload_bytes += (uint64_t)(val_off[i] - key_off[i]) + val_len[i];
  h->has_partition = partition != nullptr;
  h->n += n;
  h->kv_bytes = base + kv_bytes;
  TG_API_END
}

int32_t tezgpu_sorter_collect_fixed(tezgpu_sorter *h, const uint8_t *kv, const int32_t *partition, uint64_t n) {
  TG_API_BEGIN
  TG_CHECK(h, TEZGPU_E_INVALID, "null handle");
  TG_CHECK(!h->flushed, TEZGPU_E_STATE, "collect after flush");
  TG_CHECK(h->fixed, TEZGPU_E_STATE, "handle is not in fixed-width mode");
  if (n == 0) return TEZGPU_OK;
  TG_CHECK(kv, TEZGPU_E_INVALID, "null argument");
  TG_CHECK(h->n + n <= RADIX_MAX_N, TEZGPU_E_INVALID, "more than 2^30-1 records collected");
  TG_CHECK((h->n == 0) || (h->has_partition == (partition != nullptr)), TEZGPU_E_INVALID,
           "partition ids must be given for all batches or none");
  TG_CHECK(partition || h->pipe.conf.partitioner == TEZGPU_PART_HASH, TEZGPU_E_INVALID,
           "partition ids required (partitioner=GIVEN)");
  const uint64_t stride = (uint64_t)h->klen + h->vlen;
  {
    const uint64_t budget = h->pipe.conf.mem_budget_bytes;
    TG_CHECK(budget == 0 || h->n == 0 || (h->n + n) * stride <= budget, TEZGPU_E_NOMEM,
             "sort memory budget exceeded (" + std::to_string((h->n + n) * stride) + " > " + std::to_string(budget) +
                 " bytes): spill (flush + reset) before collecting more");
  }
  cudaStream_t st = h->pipe.stream;
  TG_CUDA(cudaSetDevice(h->pipe.conf.device));
  h->d_kv.grow_preserve((h->n + n) * stride + 32, h->n * stride, st);
  if (partition) h->d_part.grow_preserve((h->n + n) * 4, h->n * 4, st);
  TG_CUDA(cudaMemcpyAsync(h->d_kv.as<uint8_t>() + h->n * stride, kv, n * stride, cudaMemcpyHostToDevice, st));
  if (partition)
    TG_CUDA(cudaMemcpyAsync(h->d_part.as<int32_t>() + h->n, partition, n * 4, cudaMemcpyHostToDevice, st));
  TG_CUDA(cudaStreamSynchronize(st));
  h->has_partition = partition != nullptr;
  h->n += n;
  h->kv_bytes = h->n * stride;
  h->payload_bytes = h->kv_bytes;
  TG_API_END
}

uint64_t tezgpu_sorter_output_bound(const tezgpu_sorter *h) {
  if (!h) return 0;
  if (h->fixed && h->pipe.conf.rle_policy == TEZGPU_RLE_OFF)  // exact: n * (vint(k) + vint(v) + k + v) + 10 bytes per segment
    return h->n * ((uint64_t)vint_size_u32(h->klen) + vint_size_u32(h->vlen) + h->klen + h->vlen) +
           10ull * h->pipe.conf.num_partitions + 64;
  return SortPipeline::output_bound(h->n, h->kv_bytes, h->pipe.conf.num_partitions);
}

static void sorter_run(tezgpu_sorter *h, uint8_t *host_out, uint64_t out_cap, uint64_t *out_len, int64_t *index,
                       tezgpu_stats *stats, std::vector<int64_t> &idx_store) {
  TG_CHECK(!h->flushed, TEZGPU_E_STATE, "flush called twice");
  const int P = h->pipe.conf.num_partitions;
  idx_store.assign((size_t)P * 3, 0);
  uint64_t bound = tezgpu_sorter_output_bound(h);
  h->d_out.ensure(bound);
  uint64_t len = 0;
  tezgpu_stats st;
  h->pipe.run(h->records(), h->d_out.as<uint8_t>(), h->d_out.cap, &len, idx_store.data(), &st);
  st.output_bytes = (int64_t)h->payload_bytes;
  TG_CHECK(len <= out_cap, TEZGPU_E_NOMEM, "output buffer too small for file.out");
  if (len) {
    // one copy, not pieces: with 64 MB pieces a download running next to another task slot's upload was measured at
    // 26 GB/s (312 ms) instead of 40-47 GB/s (tools/e2e_probe.py, profiles/r02_e2e_probe*.log)
    TG_CUDA(cudaMemcpyAsync(host_out, h->d_out.p, len, cudaMemcpyDeviceToHost, h->pipe.stream));
    TG_CUDA(cudaStreamSynchronize(h->pipe.stream));
  }
  if (out_len) *out_len = len;
  if (index) memcpy(index, idx_store.data(), (size_t)P * 24);
  if (stats) *stats = st;
  h->flushed = true;
}

int32_t tezgpu_sorter_flush_to_memory(tezgpu_sorter *h, uint8_t *out, uint64_t out_cap, uint64_t *out_len,
                                      uint8_t *index_out, int64_t *index, tezgpu_stats *stats) {
  TG_API_BEGIN
  TG_CHECK(h && (out || out_cap == 0), TEZGPU_E_INVALID, "null argument");
  std::vector<int64_t> idx;
  sorter_run(h, out, out_cap, out_len, index, stats, idx);
  if (index_out) {
    std::vector<uint8_t> b;
    spill_record_bytes(idx.data(), h->pipe.conf.num_partitions, b);
    memcpy(index_out, b.data(), b.size());
  }
  TG_API_END
}

int32_t tezgpu_sorter_flush(tezgpu_sorter *h, const char *out_path, const char *index_path, int64_t *index,
                            tezgpu_stats *stats) {
  TG_API_BEGIN
  TG_CHECK(h && out_path && index_path, TEZGPU_E_INVALID, "null argument");
  uint64_t bound = tezgpu_sorter_output_bound(h);
  h->h_out.ensure(bound);
  std::vector<int64_t> idx;
  uint64_t len = 0;
  sorter_run(h, h->h_out.as<uint8_t>(), h->h_out.cap, &len, index, stats, idx);
  write_file_0640(out_path, h->h_out.p, len);
  std::vector<uint8_t> b;
  spill_record_bytes(idx.data(), h->pipe.conf.num_partitions, b);
  write_file_0640(index_path, b.data(), b.size());
  TG_API_END
}

int32_t tezgpu_sorter_sort_device_fixed(tezgpu_sorter *h, const void *d_kv, const void *d_partition, uint64_t n,
                                        void *d_out, uint64_t out_cap, uint64_t *out_len, int64_t *index,
                                        tezgpu_stats *stats) {
  TG_API_BEGIN
  TG_CHECK(h && (d_kv || n == 0) && d_out, TEZGPU_E_INVALID, "null argument");
  TG_CHECK(h->fixed, TEZGPU_E_STATE, "handle is not in fixed-width mode");
  TG_CHECK(n <= RADIX_MAX_N, TEZGPU_E_INVALID, "more than 2^30-1 records in one sort");
  TG_CHECK(d_partition || h->pipe.conf.partitioner == TEZGPU_PART_HASH, TEZGPU_E_INVALID,
           "partition ids required (partitioner=GIVEN)");
  Records r;
  memset(&r, 0, sizeof(r));
  r.kv = (const uint8_t *)d_kv;
  r.kv_bytes = n * ((uint64_t)h->klen + h->vlen);  // exact: boundary loads are clamped, nothing is read past the caller's buffer
  r.partition = (const int32_t *)d_partition;
  r.n = (uint32_t)n;
  r.klen = h->klen;
  r.vlen = h->vlen;
  r.fixed = 1;
  TG_CHECK(((uintptr_t)d_kv & 15u) == 0, TEZGPU_E_INVALID, "device-resident input must be 16-byte aligned");
  tezgpu_stats st;
  h->pipe.run(r, (uint8_t *)d_out, out_cap, out_len, index, &st);
  st.output_bytes = (int64_t)(n * ((uint64_t)h->klen + h->vlen));
  if (stats) *stats = st;
  TG_API_END
}

void *tezgpu_sorter_stream(tezgpu_sorter *h) { return h ? (void *)h->pipe.stream : nullptr; }

int32_t tezgpu_sorter_set_combiner(tezgpu_sorter *h, int32_t kind) {
  TG_API_BEGIN
  TG_CHECK(h, TEZGPU_E_INVALID, "null handle");
  TG_CHECK(kind >= TEZGPU_COMBINE_NONE && kind <= TEZGPU_COMBINE_LONG_SUM, TEZGPU_E_INVALID, "unknown combiner kind");
  TG_CHECK(h->n == 0 && !h->flushed, TEZGPU_E_STATE, "set the combiner before the first collect or right after a reset");
  TG_CHECK(kind == TEZGPU_COMBINE_NONE || h->pipe.conf.sorter_impl != TEZGPU_SORTER_UNORDERED, TEZGPU_E_UNSUPPORTED,
           "an unordered output has no combiner (its records are not grouped by key)");
  const uint32_t vw = kind == TEZGPU_COMBINE_INT_SUM ? 4 : 8;
  TG_CHECK(kind == TEZGPU_COMBINE_NONE || h->pipe.conf.fixed_val_len == 0 || h->pipe.conf.fixed_val_len == vw, TEZGPU_E_INVALID,
           "fixed_val_len " + std::to_string(h->pipe.conf.fixed_val_len) + " is not the combiner's value width (" +
               std::to_string(vw) + " bytes)");
  h->pipe.combine_kind = kind;
  TG_API_END
}

int32_t tezgpu_sorter_combine_info(tezgpu_sorter *h, uint64_t *records_in, uint64_t *records_out, float *ms) {
  TG_API_BEGIN
  TG_CHECK(h, TEZGPU_E_INVALID, "null handle");
  if (records_in) *records_in = h->pipe.combine_in;
  if (records_out) *records_out = h->pipe.combine_out;
  if (ms) *ms = h->pipe.combine_ms;
  TG_API_END
}

// ------------------------------------------------------------------------------------------------ NVLink peer fetch
int32_t tezgpu_peer_alloc(int32_t device, uint64_t bytes, void **dptr, uint8_t *handle_out) {
  TG_API_BEGIN
  TG_CHECK(dptr && handle_out && bytes, TEZGPU_E_INVALID, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == TEZGPU_PEER_HANDLE_BYTES, "export handle size");
  TG_CUDA(cudaSetDevice(device));
  void *p = nullptr;
  TG_CUDA(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    TG_CUDA(e);
  }
  memcpy(handle_out, &h, sizeof(h));
  *dptr = p;
  TG_API_END
}

int32_t tezgpu_peer_free(int32_t device, void *dptr) {
  TG_API_BEGIN
  TG_CUDA(cudaSetDevice(device));
  if (dptr) TG_CUDA(cudaFree(dptr));
  TG_API_END
}

int32_t tezgpu_peer_open(int32_t device, const uint8_t *handle, void **dptr) {
  TG_API_BEGIN
  TG_CHECK(handle && dptr, TEZGPU_E_INVALID, "null argument");
  TG_CUDA(cudaSetDevice(device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void *p = nullptr;
  TG_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  *dptr = p;
  TG_API_END
}

int32_t tezgpu_peer_close(int32_t device, void *dptr) {
  TG_API_BEGIN
  TG_CUDA(cudaSetDevice(device));
  if (dptr) TG_CUDA(cudaIpcCloseMemHandle(dptr));
  TG_API_END
}

}  // extern "C"
// TEZGPU_FETCH_CTAS (read at every call): upper bound on the pull kernels' grid.  The pull is NVLink-bound; when it runs
// next to another stream's HBM-bound kernels (TEZ_SHUFFLE_OVERLAP: the sort of the next batch) a grid that fills every
// SM makes the two serialise, a grid of about one CTA per SM leaves room for the other kernels' CTAs.
static uint32_t fetch_grid_cap(uint32_t grid) {
  const char *e = getenv("TEZGPU_FETCH_CTAS");
  const long cap = e ? atol(e) : 0;
  return cap > 0 && (uint32_t)cap < grid ? (uint32_t)cap : grid;
}
extern "C" {
int32_t tezgpu_fetch_ranges(int32_t device, const tezgpu_copy_range *ranges, uint32_t n, void *stream, float *ms_kernel) {
  TG_API_BEGIN
  TG_CHECK(ranges || n == 0, TEZGPU_E_INVALID, "null argument");
  if (ms_kernel) *ms_kernel = 0;
  if (n == 0) return TEZGPU_OK;
  TG_CUDA(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<FetchRange> fr(n);
  uint64_t chunks = 0;
  for (uint32_t i = 0; i < n; i++) {
    TG_CHECK((ranges[i].src && ranges[i].dst) || ranges[i].len == 0, TEZGPU_E_INVALID, "null range");
    fr[i].src = (const uint8_t *)ranges[i].src;
    fr[i].dst = (uint8_t *)ranges[i].dst;
    fr[i].len = ranges[i].len;
    fr[i].chunk0 = chunks;
    chunks += fetch_chunks(ranges[i].src, ranges[i].dst, ranges[i].len);
  }
  if (chunks == 0) return TEZGPU_OK;
  // ranges travel as a kernel parameter when they are few (one per peer GPU); larger lists through a device copy
  FetchRange *d_fr = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  cudaError_t err = cudaSuccess;
  if (n > FETCH_INLINE_RANGES) {
    TG_CUDA(cudaMalloc(&d_fr, (size_t)n * sizeof(FetchRange)));
    err = cudaMemcpyAsync(d_fr, fr.data(), (size_t)n * sizeof(FetchRange), cudaMemcpyHostToDevice, st);
  }
  if (err == cudaSuccess && ms_kernel) {
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, st);
  }
  if (err == cudaSuccess) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    uint32_t grid = (uint32_t)std::min<uint64_t>(chunks, (uint64_t)sms * 2);
    grid = fetch_grid_cap(grid);
    if (d_fr) {
      k_fetch_ranges<<<grid, FETCH_THREADS, 0, st>>>(d_fr, n, chunks);
    } else {
      FetchRangeList lst;
      for (uint32_t i = 0; i < n; i++) lst.r[i] = fr[i];
      k_fetch_ranges_inline<<<grid, FETCH_THREADS, 0, st>>>(lst, n, chunks);
    }
    err = cudaGetLastError();
  }
  if (err == cudaSuccess && ms_kernel) cudaEventRecord(e1, st);
  if (err == cudaSuccess) err = cudaStreamSynchronize(st);
  if (err == cudaSuccess && ms_kernel) cudaEventElapsedTime(ms_kernel, e0, e1);
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  if (d_fr) cudaFree(d_fr);
  TG_CUDA(err);
  TG_API_END
}

// per-device scratch of tezgpu_fetch_ranges_verified (grow-only; one fetch at a time per device)
struct FetchVerifyScratch {
  DeviceBuffer segs, piece_start, piece_crc, seg_crc, flag;
  std::mutex mu;
};
static FetchVerifyScratch &fetch_scratch(int device) {
  static FetchVerifyScratch inst[64];
  return inst[device & 63];
}

int32_t tezgpu_fetch_segments_verified(int32_t device, const tezgpu_fetch_segment *segs, uint32_t n, void *stream,
                                       float *ms_kernel) {
  TG_API_BEGIN
  TG_CHECK(segs || n == 0, TEZGPU_E_INVALID, "null argument");
  if (ms_kernel) *ms_kernel = 0;
  if (n == 0) return TEZGPU_OK;
  TG_CUDA(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<FetchSeg> fs(n);
  std::vector<uint32_t> piece_start(n + 1);
  uint32_t np = 0;
  for (uint32_t i = 0; i < n; i++) {
    const bool hdr = segs[i].flags & TEZGPU_SEG_HAS_HEADER;
    TG_CHECK(segs[i].src && segs[i].dst, TEZGPU_E_INVALID, "null segment");
    TG_CHECK(segs[i].len >= (hdr ? 10u : 6u), TEZGPU_E_FORMAT, "IFile segment shorter than an empty segment");
    TG_CHECK((((uintptr_t)segs[i].src ^ (uintptr_t)segs[i].dst) & 15u) == 0, TEZGPU_E_INVALID,
             "source and destination of a verified fetch must agree modulo 16");
    fs[i].src = (const uint8_t *)segs[i].src;
    fs[i].dst = (uint8_t *)segs[i].dst;
    fs[i].len = segs[i].len;
    fs[i].has_header = hdr ? 1 : 0;
    fs[i].pad = 0;
    piece_start[i] = np;
    np += (uint32_t)div_up(segs[i].len - 4 - (hdr ? 4 : 0), FV_PIECE);
  }
  piece_start[n] = np;
  FetchVerifyScratch &sc = fetch_scratch(device);
  std::lock_guard<std::mutex> lock(sc.mu);
  sc.segs.ensure((size_t)n * sizeof(FetchSeg));
  sc.piece_start.ensure((size_t)(n + 1) * 4);
  sc.piece_crc.ensure((size_t)np * sizeof(TileCrc));
  sc.seg_crc.ensure((size_t)n * 4);
  sc.flag.ensure(16);
  const CrcTables *d_crc = DeviceConstants::get(device).d_crc;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  TG_CUDA(cudaMemcpyAsync(sc.segs.p, fs.data(), (size_t)n * sizeof(FetchSeg), cudaMemcpyHostToDevice, st));
  TG_CUDA(cudaMemcpyAsync(sc.piece_start.p, piece_start.data(), (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, st));
  TG_CUDA(cudaMemsetAsync(sc.seg_crc.p, 0, (size_t)n * 4, st));
  TG_CUDA(cudaMemsetAsync(sc.flag.p, 0, 16, st));
  if (ms_kernel) {
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, st);
  }
  int sms = 148, per_sm = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fetch_verify, FV_THREADS, 0);
  const uint32_t grid = fetch_grid_cap((uint32_t)std::min<uint64_t>(np, (uint64_t)sms * (per_sm > 0 ? per_sm : 1)));
  k_fetch_verify<<<grid, FV_THREADS, 0, st>>>(sc.segs.as<FetchSeg>(), sc.piece_start.as<uint32_t>(), n, np, d_crc, sc.piece_crc.as<TileCrc>());
  if (ms_kernel) cudaEventRecord(e1, st);
  k_crc_combine<<<(uint32_t)div_up(np, 256), 256, 0, st>>>(sc.piece_crc.as<TileCrc>(), np, d_crc, sc.seg_crc.as<uint32_t>());
  k_fetch_crc_check<<<(uint32_t)div_up(n, 128), 128, 0, st>>>(sc.segs.as<FetchSeg>(), n, sc.seg_crc.as<uint32_t>(), d_crc, sc.flag.as<int>());
  cudaError_t err = cudaGetLastError();
  int bad = 0;
  if (err == cudaSuccess) err = cudaMemcpyAsync(&bad, sc.flag.p, 4, cudaMemcpyDeviceToHost, st);
  if (err == cudaSuccess) err = cudaStreamSynchronize(st);
  if (err == cudaSuccess && ms_kernel) cudaEventElapsedTime(ms_kernel, e0, e1);
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  TG_CUDA(err);
  TG_CHECK(bad == 0, TEZGPU_E_FORMAT, "IFile checksum mismatch in fetched segment " + std::to_string(bad - 1));
  TG_API_END
}

#include "shuffle_wire.inl"

// Host emulation of the emit kernel's parallel CRC scheme (interleaved per-thread streams over the 4-byte words of a
// piece, power-table alignment, xor-fold of piece contributions into the segment remainder, final conditioning).
// Pure host arithmetic on the same tables the device uses; lets the CPU test-suite check the GF(2) algebra.
uint32_t tezgpu_debug_crc_emulate(const uint8_t *body, uint64_t len, uint32_t piece_bytes, uint32_t lead) {
  CrcTables *t = new CrcTables();
  const int T = EMIT_CRC_STRIDE_WORDS;
  crc_build_tables(*t, T);
  auto shift = [&](uint32_t crc, uint64_t nbytes) {
    uint32_t a0 = (uint32_t)(nbytes & 4095), a1 = (uint32_t)((nbytes >> 12) & 4095), a2 = (uint32_t)((nbytes >> 24) & 4095);
    if (a0) crc = crc_multmodp(crc, t->pow0[a0]);
    if (a1) crc = crc_multmodp(crc, t->pow1[a1]);
    if (a2) crc = crc_multmodp(crc, t->pow2[a2]);
    return crc;
  };
  uint32_t seg = 0;
  uint64_t done = 0;
  std::vector<uint8_t> img;
  while (done < len) {
    uint32_t ld = (uint32_t)((done + lead) & 15u);
    uint32_t plen = (uint32_t)std::min<uint64_t>(piece_bytes - ld, len - done);
    img.assign((size_t)ld + plen + 16, 0);
    memcpy(img.data() + ld, body + done, plen);
    uint32_t cb0 = ld, cb1 = ld + plen;
    uint32_t wa = (cb0 + 3u) >> 2, wb = cb1 >> 2;
    uint32_t words_crc = 0;
    const uint32_t *img32 = reinterpret_cast<const uint32_t *>(img.data());
    if (wb > wa) {
      uint32_t W = wb - wa;
      for (uint32_t tid = 0; tid < (uint32_t)T && tid < W; tid++) {
        uint32_t i = wa + tid, c = 0;
        for (; i + T < wb; i += T) {
          uint32_t v = c ^ img32[i];
          c = t->adv[0][v & 0xFF] ^ t->adv[1][(v >> 8) & 0xFF] ^ t->adv[2][(v >> 16) & 0xFF] ^ t->adv[3][v >> 24];
        }
        uint32_t v = c ^ img32[i];
        c = t->slice[3][v & 0xFF] ^ t->slice[2][(v >> 8) & 0xFF] ^ t->slice[1][(v >> 16) & 0xFF] ^ t->slice[0][v >> 24];
        uint32_t d = wb - 1 - i;
        if (d) c = crc_multmodp(c, t->pow_word[d]);
        words_crc ^= c;
      }
    }
    uint32_t raw = 0;
    uint32_t head_end = (wb > wa) ? 4 * wa : cb1;
    for (uint32_t b = cb0; b < head_end; b++) raw = t->slice[0][(raw ^ img[b]) & 0xFF] ^ (raw >> 8);
    if (wb > wa) {
      raw = shift(raw, 4ull * (wb - wa)) ^ words_crc;
      for (uint32_t b = 4 * wb; b < cb1; b++) raw = t->slice[0][(raw ^ img[b]) & 0xFF] ^ (raw >> 8);
    }
    seg ^= shift(raw, len - (done + plen));
    done += plen;
  }
  uint32_t crc = seg ^ shift(0xFFFFFFFFu, len) ^ 0xFFFFFFFFu;
  delete t;
  return crc;
}

// Host emulation of the TMA emit kernel's chunk assembly (emit_tma.cuh): builds the output byte image of one tile chunk
// by chunk with the very same template code the consumer warps run, from `nr` staged records of `stride` bytes.
// image_out receives 16 * (chunks) bytes starting at image offset 0; returns the image length (body_end).
uint32_t tezgpu_debug_assemble_emulate(const uint8_t *stage, uint32_t nr, uint32_t stride, const uint8_t *hdr, uint32_t hdr_len,
                                       uint32_t lead, int32_t first, int32_t last, uint8_t *image_out, uint32_t image_cap) {
  std::vector<uint8_t> padded((size_t)nr * stride + 64, 0);
  memcpy(padded.data(), stage, (size_t)nr * stride);
  HostSmem sm{padded.data()};
  TmaEmitConst kc;
  kc.rec_size = hdr_len + stride;
  kc.hdr_len = hdr_len;
  kc.stride = stride;
  kc.magic = (uint32_t)((1ull << 32) / kc.rec_size) + 1u;
  uint32_t hw[4] = {0, 0, 0, 0};
  for (uint32_t b = 0; b < hdr_len; b++) hw[b >> 2] |= (uint32_t)hdr[b] << (8u * (b & 3u));
  kc.hdr = make_uint4(hw[0], hw[1], hw[2], hw[3]);
  TmaTileGeom g;
  g.stg = 0;
  g.nr = nr;
  g.first = first != 0;
  g.last = last != 0;
  g.rec0 = lead + (g.first ? 4u : 0u);
  g.body = nr * kc.rec_size;
  const uint32_t body_end = g.rec0 + g.body + (g.last ? 2u : 0u);
  for (uint32_t c = lead >> 4; 16u * c < body_end && 16u * c + 16u <= image_cap; c++) {
    const uint4 v = tma_assemble(sm, kc, g, 16u * c);
    memcpy(image_out + 16u * c, &v, 16);
  }
  return body_end;
}

// Host emulation of the chunk-interleaved checksum of the emit / verify kernels (crc32.cuh CrcChunkFold): 256 threads,
// thread t folds chunks i = Cn + t - iters*256 (+256 ...), partials are combined by the adv128 second-level fold, the
// per-lane alignment multiplier and an xor across lanes.  ilp = 1 runs the two-deep fold with the einv correction,
// ilp = 0 the textbook chain.  Returns the raw remainder (init 0, no final xor) of the nchunks * 16 bytes.
uint32_t tezgpu_debug_chunk_fold_emulate(const uint8_t *data, uint32_t nchunks, int32_t ilp) {
  CrcTables *t = new CrcTables();
  const int T = EMIT_CRC_STRIDE_WORDS;
  crc_build_tables(*t, T);
  auto tab = [](const uint32_t(*m)[256], uint32_t x) { return m[0][x & 0xFF] ^ m[1][(x >> 8) & 0xFF] ^ m[2][(x >> 16) & 0xFF] ^ m[3][x >> 24]; };
  auto W = [&](uint32_t x) { return t->slice[3][x & 0xFF] ^ t->slice[2][(x >> 8) & 0xFF] ^ t->slice[1][(x >> 16) & 0xFF] ^ t->slice[0][x >> 24]; };
  auto S = [&](uint32_t x) { return tab(t->advc, x); };
  auto SW2 = [&](uint32_t x) { return tab(t->advc2, x); };
  const uint32_t Cn = nchunks, iters = (Cn + T - 1) / T;
  std::vector<uint32_t> part(T, 0);
  for (int tid = 0; tid < T; tid++) {
    int64_t i = (int64_t)Cn + tid - (int64_t)iters * T;
    uint32_t c = 0;
    for (uint32_t it = 0; it < iters; it++, i += T) {
      uint32_t w[4] = {0, 0, 0, 0};
      if (i >= 0) memcpy(w, data + 16 * i, 16);
      if (ilp) {
        const uint32_t u = W(c ^ w[0]) ^ w[1], r = W(w[2]) ^ w[3];
        c = SW2(u) ^ S(r);
      } else {
        uint32_t x = W(c ^ w[0]) ^ w[1];
        x = W(x) ^ w[2];
        x = W(x) ^ w[3];
        c = (it + 1 == iters) ? W(x) : S(x);
      }
    }
    part[tid] = c;
  }
  uint32_t total = 0;
  for (int lane = 0; lane < 32; lane++) {
    uint32_t q = 0;
    for (int kk = 0; kk < T / 32; kk++) q = tab(t->adv128, q) ^ part[lane + 32 * kk];
    uint32_t lp = t->pow_word[4 * (31 - lane)];
    if (ilp) lp = crc_multmodp(lp, t->einv);
    total ^= crc_multmodp(q, lp);
  }
  // the identity the correction rests on: einv * x^(128*(T-1)) == 1
  if (crc_multmodp(t->einv, crc_host_xpow8((uint64_t)16 * (uint64_t)(T - 1))) != 0x80000000u) total = ~total;
  delete t;
  return total;
}

// Host emulation of the run-range emit kernel's chunk assembly (emit_runs.cuh): record j of the tile is the rec_size
// bytes at staging[src[j]...]; builds the output image chunk by chunk with the kernel's template code.
uint32_t tezgpu_debug_runs_assemble_emulate(const uint8_t *staging, uint32_t staging_len, const uint32_t *src, uint32_t nr,
                                            uint32_t rec_size, uint32_t lead, int32_t first, int32_t last, uint8_t *image_out,
                                            uint32_t image_cap) {
  std::vector<uint8_t> padded((size_t)staging_len + 64, 0);
  memcpy(padded.data(), staging, staging_len);
  HostSmem sm{padded.data()};
  RunsTileGeom g;
  g.src = src;
  g.nr = nr;
  g.first = first != 0;
  g.last = last != 0;
  g.rec0 = lead + (g.first ? 4u : 0u);
  g.body = nr * rec_size;
  const uint32_t magic = (uint32_t)((1ull << 32) / rec_size) + 1u;
  const uint32_t body_end = g.rec0 + g.body + (g.last ? 2u : 0u);
  for (uint32_t c = lead >> 4; 16u * c < body_end && 16u * c + 16u <= image_cap; c++) {
    const uint4 v = runs_assemble(sm, rec_size, magic, g, 16u * c);
    memcpy(image_out + 16u * c, &v, 16);
  }
  return body_end;
}

}  // extern "C"

#include "merger_api.inl"
