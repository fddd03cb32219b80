// tez_runtime_library.cc -- host-side C++ mirror of OrderedPartitionedKVOutput / OrderedGroupedKVInput on top of the
// tezgpu_* C ABI (include/tezgpu.h).  See include/tez_runtime.h.  Host logic only: configuration, memory request,
// spill policy, file naming, counters, events, value grouping.  All sorting / merging / IFile bytes come from the
// device library -- there is no CPU implementation of the hot path in here.
//
// RL/  = /root/reference/tez-runtime-library/src/main/java/org/apache/tez/runtime/library/
// SORT/ = RL/common/sort/impl/   OG/ = RL/common/shuffle/orderedgrouped/
#include <errno.h>
#include <fcntl.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../../include/tez_runtime.h"
#include "../../../include/tezgpu.h"

namespace tezrt {

struct Err : std::runtime_error {
  int code;
  Err(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};
static thread_local std::string g_err;
#define RT_CHECK(cond, code, msg) do { if (!(cond)) throw Err((code), (msg)); } while (0)
static void gpu_check(int32_t rc) { if (rc != 0) throw Err(rc, tezgpu_last_error()); }

// ---------------------------------------------------------------- configuration (keys: RL/api/TezRuntimeConfiguration.java)
struct Configuration {
  std::map<std::string, std::string> kv;
  explicit Configuration(const char *text) {
    std::string s = text ? text : "";
    size_t pos = 0;
    while (pos < s.size()) {
      size_t nl = s.find('\n', pos);
      if (nl == std::string::npos) nl = s.size();
      std::string line = s.substr(pos, nl - pos);
      size_t eq = line.find('=');
      if (eq != std::string::npos) kv[line.substr(0, eq)] = line.substr(eq + 1);
      pos = nl + 1;
    }
  }
  std::string get(const std::string &k, const std::string &d) const { auto it = kv.find(k); return it == kv.end() ? d : it->second; }
  long getInt(const std::string &k, long d) const { auto it = kv.find(k); return it == kv.end() ? d : atol(it->second.c_str()); }
  double getFloat(const std::string &k, double d) const { auto it = kv.find(k); return it == kv.end() ? d : atof(it->second.c_str()); }
  bool getBoolean(const std::string &k, bool d) const {
    auto it = kv.find(k);
    if (it == kv.end()) return d;
    return it->second == "true" || it->second == "TRUE" || it->second == "1";
  }
};

static const char *K_SORT_MB = "tez.runtime.io.sort.mb";                       // :115-116 default 100
static const char *K_SORTER_CLASS = "tez.runtime.sorter.class";                // :167-169 default PIPELINED
static const char *K_KEY_CLASS = "tez.runtime.key.class";
static const char *K_KEY_COMPARATOR = "tez.runtime.key.comparator.class";
static const char *K_PARTITIONER = "tez.runtime.partitioner.class";
static const char *K_EMPTY_PARTITIONS = "tez.runtime.empty.partitions.info-via-events.enabled";  // :506-509 default true
static const char *K_FINAL_MERGE = "tez.runtime.enable.final-merge.in.output";  // :555-557 default true
static const char *K_REPORT_STATS = "tez.runtime.report.partition.stats";       // :195-198 default memory_optimized
static const char *K_COMPRESS = "tez.runtime.compress";
static const char *K_SERIALIZATIONS = "io.serializations";
static const char *K_VALUE_CLASS = "tez.runtime.value.class";
static const char *K_COMBINER = "tez.runtime.combiner.class";
static const char *K_COMBINE_MIN_SPILLS = "tez.runtime.combine.min.spills";  // :128-130 default 3

static bool ends_with(const std::string &s, const char *suf) {
  size_t n = strlen(suf);
  return s.size() >= n && s.compare(s.size() - n, n, suf) == 0;
}

// closed set of key classes the device can order (SURVEY 7 "hard parts"); anything else is rejected at start()
static int comparator_for(const Configuration &c) {
  std::string key = c.get(K_KEY_CLASS, ""), cmp = c.get(K_KEY_COMPARATOR, ""), ser = c.get(K_SERIALIZATIONS, "");
  if (ends_with(key, "io.Text")) return TEZGPU_CMP_TEXT;
  if (ends_with(key, "io.IntWritable")) return TEZGPU_CMP_INT;
  if (ends_with(key, "io.LongWritable")) return TEZGPU_CMP_LONG;
  if (ends_with(key, "io.BytesWritable")) {
    if (ends_with(cmp, "TezBytesComparator") || ser.find("TezBytesWritableSerialization") != std::string::npos) return TEZGPU_CMP_BYTES;
    return TEZGPU_CMP_BYTESWRITABLE;
  }
  throw Err(TEZGPU_E_UNSUPPORTED, "key class '" + key + "' has no device comparator (supported: Text, BytesWritable, IntWritable, LongWritable)");
}

// MRCombiner over a sum reducer runs on the device (TEZGPU_COMBINE_*).  MRCombiner takes the reducer class from
// mapreduce.job.combine.class under the new API and from mapred.combiner.class otherwise (ConfigUtils.useNewApi,
// RL/common/ConfigUtils.java:128-130).  Any other combiner class is not run, as before the device combiner existed.
static int combiner_for(const Configuration &c) {
  if (c.get(K_COMBINER, "") != "org.apache.tez.mapreduce.combine.MRCombiner") return TEZGPU_COMBINE_NONE;
  const bool new_api = c.getBoolean("mapred.mapper.new-api", false);
  const std::string red = c.get(new_api ? "mapreduce.job.combine.class" : "mapred.combiner.class", "");
  int kind;
  std::string need;
  if (red == "org.apache.hadoop.mapreduce.lib.reduce.IntSumReducer") {
    kind = TEZGPU_COMBINE_INT_SUM;
    need = "org.apache.hadoop.io.IntWritable";
  } else if (red == "org.apache.hadoop.mapreduce.lib.reduce.LongSumReducer" || red == "org.apache.hadoop.mapred.lib.LongSumReducer") {
    kind = TEZGPU_COMBINE_LONG_SUM;
    need = "org.apache.hadoop.io.LongWritable";
  } else {
    return TEZGPU_COMBINE_NONE;
  }
  // the reference would fail later, at the first spill, with a ClassCastException inside the reducer
  const std::string val = c.get(K_VALUE_CLASS, "");
  RT_CHECK(val == need, TEZGPU_E_UNSUPPORTED, "combiner " + red + " sums " + need + " values, but the value class is '" + val + "'");
  return kind;
}

// ---------------------------------------------------------------- small utilities
static void mkdirs(const std::string &path) {
  for (size_t i = 1; i <= path.size(); i++)
    if (i == path.size() || path[i] == '/') {
      std::string p = path.substr(0, i);
      if (::mkdir(p.c_str(), 0755) != 0 && errno != EEXIST) throw Err(TEZGPU_E_IO, "mkdir " + p + ": " + strerror(errno));
    }
}
static std::vector<uint8_t> read_file(const std::string &p, uint64_t off = 0, int64_t len = -1) {
  int fd = ::open(p.c_str(), O_RDONLY);
  RT_CHECK(fd >= 0, TEZGPU_E_IO, "open " + p + ": " + strerror(errno));
  struct stat st;
  fstat(fd, &st);
  uint64_t n = len < 0 ? (uint64_t)st.st_size - off : (uint64_t)len;
  std::vector<uint8_t> b(n);
  uint64_t got = 0;
  while (got < n) {
    ssize_t r = ::pread(fd, b.data() + got, n - got, (off_t)(off + got));
    if (r <= 0) { ::close(fd); throw Err(TEZGPU_E_IO, "short read of " + p); }
    got += (uint64_t)r;
  }
  ::close(fd);
  return b;
}
// TezCommonUtils.compressByteArrayToByteString with newBestCompressionDeflater(): raw deflate, level 9
static std::string deflate_raw(const std::vector<uint8_t> &in) {
  z_stream z;
  memset(&z, 0, sizeof(z));
  RT_CHECK(deflateInit2(&z, 9, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) == Z_OK, TEZGPU_E_INVALID, "deflateInit2");
  std::string out(deflateBound(&z, in.size()) + 16, '\0');
  z.next_in = const_cast<Bytef *>(in.data());
  z.avail_in = (uInt)in.size();
  z.next_out = (Bytef *)&out[0];
  z.avail_out = (uInt)out.size();
  int rc = deflate(&z, Z_FINISH);
  RT_CHECK(rc == Z_STREAM_END, TEZGPU_E_INVALID, "deflate");
  out.resize(z.total_out);
  deflateEnd(&z);
  return out;
}
// protobuf wire helpers (ShufflePayloads.proto)
static void pb_varint(std::string &o, uint64_t v) { while (v >= 0x80) { o.push_back((char)(v | 0x80)); v >>= 7; } o.push_back((char)v); }
static void pb_tag(std::string &o, int field, int wt) { pb_varint(o, (uint64_t)(field << 3 | wt)); }
static void pb_bytes(std::string &o, int field, const std::string &b) { pb_tag(o, field, 2); pb_varint(o, b.size()); o += b; }
static void pb_int(std::string &o, int field, int64_t v) { pb_tag(o, field, 0); pb_varint(o, (uint64_t)v); }

struct Event {
  int type;
  std::string payload;
  int source_index_start = 0, count = 0;
};

// RoaringBitmap portable serialization (no run containers) of a sorted value list -- the format
// RoaringBitmap.serialize(DataOutput) writes for ShuffleUtils.getPartitionStatsForPhysicalOutput (:486-500)
static std::vector<uint8_t> roaring_serialize(const std::vector<uint32_t> &vals) {
  std::vector<std::pair<uint16_t, std::vector<uint16_t>>> cont;
  for (uint32_t v : vals) {
    uint16_t hi = (uint16_t)(v >> 16), lo = (uint16_t)v;
    if (cont.empty() || cont.back().first != hi) cont.push_back({hi, {}});
    cont.back().second.push_back(lo);
  }
  std::vector<uint8_t> o;
  auto u16 = [&](uint32_t x) { o.push_back((uint8_t)x); o.push_back((uint8_t)(x >> 8)); };
  auto u32 = [&](uint32_t x) { u16(x & 0xFFFF); u16(x >> 16); };
  u32(12346);  // SERIAL_COOKIE_NO_RUNCONTAINER
  u32((uint32_t)cont.size());
  for (auto &c : cont) { u16(c.first); u16((uint32_t)c.second.size() - 1); }
  uint32_t off = 8 + 8 * (uint32_t)cont.size();
  for (auto &c : cont) { u32(off); off += c.second.size() > 4096 ? 8192u : 2u * (uint32_t)c.second.size(); }
  for (auto &c : cont) {
    if (c.second.size() > 4096) {
      std::vector<uint8_t> bm(8192, 0);
      for (uint16_t x : c.second) bm[x >> 3] |= (uint8_t)(1u << (x & 7));
      o.insert(o.end(), bm.begin(), bm.end());
    } else {
      for (uint16_t x : c.second) u16(x);
    }
  }
  return o;
}

// ================================================================================================ output side
// GpuSorter: the ExternalSorter seam (SORT/ExternalSorter.java:74-92,281-288) backed by tezgpu_sorter.  Records are
// batched on the host and handed to the device; when the collected bytes reach the granted sort memory the device
// content is spilled (sorted IFile + index), and flush() either renames the single spill or runs the final merge over
// the spills on the device (PipelinedSorter.flush :664-859).
struct GpuSorter {
  tezgpu_sorter *h = nullptr;
  tezgpu_conf gc;
  int P;
  int64_t available_memory;
  bool final_merge;
  std::string work_dir, uid;
  // host batch
  std::vector<uint8_t> kv;
  std::vector<uint32_t> koff, voff, vlen;
  std::vector<int32_t> part;
  bool given_partitions = false;
  uint64_t collected_bytes = 0;
  int num_spills = 0;
  std::vector<std::string> spill_files, spill_index_files;
  std::vector<std::vector<int64_t>> spill_index;
  std::string final_out, final_index;
  std::vector<int64_t> final_idx;
  std::vector<int64_t> partition_stats;  // partitionStats[p] += rawLength at every spill (SORT/PipelinedSorter.java:631-633)
  int last_spill_rle = 0;                // merger.needsRLE() of the most recent spill's SpanMerger (:599,805,814)
  int combine_kind = TEZGPU_COMBINE_NONE;
  long min_spills_for_combine = 3;
  std::map<std::string, int64_t> &counters;

  GpuSorter(const tezgpu_conf &c, int64_t mem, bool fm, const std::string &wd, const std::string &u, std::map<std::string, int64_t> &ctr,
            int combiner, long min_spills)
      : gc(c), P(c.num_partitions), available_memory(mem), final_merge(fm), work_dir(wd), uid(u), combine_kind(combiner),
        min_spills_for_combine(min_spills), counters(ctr) {
    gpu_check(tezgpu_sorter_create(&gc, &h));
    if (combine_kind != TEZGPU_COMBINE_NONE) gpu_check(tezgpu_sorter_set_combiner(h, combine_kind));
  }
  // TaskCounter.COMBINE_INPUT_RECORDS / COMBINE_OUTPUT_RECORDS of one combine (ValuesIterator / the combiner's writer)
  void count_combine(uint64_t in, uint64_t out) {
    counters["COMBINE_INPUT_RECORDS"] += (int64_t)in;
    counters["COMBINE_OUTPUT_RECORDS"] += (int64_t)out;
  }
  ~GpuSorter() { if (h) tezgpu_sorter_destroy(h); }

  // TezTaskOutputFiles (RL/common/task/local/output/TezTaskOutputFiles.java:88-231)
  std::string spill_dir(int n) const { return work_dir + "/output/" + uid + "_" + std::to_string(n); }
  std::string final_dir() const { return work_dir + "/output/" + uid; }

  void push_batch() {
    if (koff.empty()) return;
    gpu_check(tezgpu_sorter_collect_batch(h, kv.data(), kv.size(), koff.data(), voff.data(), vlen.data(),
                                          given_partitions ? part.data() : nullptr, (uint32_t)koff.size()));
    kv.clear(); koff.clear(); voff.clear(); vlen.clear(); part.clear();
  }

  void write(const uint8_t *k, uint32_t kl, const uint8_t *v, uint32_t vl, int32_t partition) {
    if (partition >= 0) {
      RT_CHECK(partition < P, TEZGPU_E_INVALID, "Illegal partition for key (" + std::to_string(partition) + ")");  // PipelinedSorter.java:410-413
      RT_CHECK(given_partitions || (koff.empty() && collected_bytes == 0 && num_spills == 0), TEZGPU_E_INVALID, "mixing partitioner modes");
      given_partitions = true;
    } else {
      RT_CHECK(!given_partitions, TEZGPU_E_INVALID, "mixing partitioner modes");
    }
    uint64_t rec = (uint64_t)kl + vl;
    if (collected_bytes && collected_bytes + kv.size() + rec > (uint64_t)available_memory) { push_batch(); spill(); }
    koff.push_back((uint32_t)kv.size());
    kv.insert(kv.end(), k, k + kl);
    voff.push_back((uint32_t)kv.size());
    kv.insert(kv.end(), v, v + vl);
    vlen.push_back(vl);
    if (given_partitions) part.push_back(partition);
    counters["OUTPUT_RECORDS"]++;
    counters["OUTPUT_BYTES"] += (int64_t)rec;
    if (kv.size() >= (32u << 20) || kv.size() + 8 >= (uint64_t)available_memory) {
      collected_bytes += kv.size();
      push_batch();
    }
  }

  void spill() {
    std::string dir = spill_dir(num_spills);
    mkdirs(dir);
    std::string f = dir + "/file.out", fi = f + ".index";
    std::vector<int64_t> idx((size_t)P * 3);
    tezgpu_stats st;
    gpu_check(tezgpu_sorter_flush(h, f.c_str(), fi.c_str(), idx.data(), &st));
    if (combine_kind != TEZGPU_COMBINE_NONE) {  // runCombineProcessor per partition at every spill (:601-609)
      uint64_t in = 0, out = 0;
      gpu_check(tezgpu_sorter_combine_info(h, &in, &out, nullptr));
      count_combine(in, out);
    }
    gpu_check(tezgpu_sorter_reset(h));
    // adjustSpillCounters (:468-482)
    if (!final_merge) counters["OUTPUT_BYTES_WITH_OVERHEAD"] += st.output_bytes_with_overhead;
    else if (num_spills > 0) { counters["ADDITIONAL_SPILLS_BYTES_WRITTEN"] += st.file_out_bytes; counters["OUTPUT_BYTES_WITH_OVERHEAD"] = 0; }
    else counters["OUTPUT_BYTES_WITH_OVERHEAD"] += st.output_bytes_with_overhead;
    counters["SPILLED_RECORDS"] += st.spilled_records;
    last_spill_rle = st.rle_used;
    partition_stats.resize((size_t)P, 0);
    for (int p = 0; p < P; p++) partition_stats[p] += idx[3 * p + 1];
    spill_files.push_back(f);
    spill_index_files.push_back(fi);
    spill_index.push_back(idx);
    num_spills++;
    collected_bytes = 0;
  }

  void flush() {
    collected_bytes += kv.size();
    push_batch();
    spill();  // "force a spill in flush()" (:679-690)
    counters["ADDITIONAL_SPILL_COUNT"] += num_spills - 1;
    if (!final_merge) {
      counters["SHUFFLE_CHUNK_COUNT"] = num_spills;
      int64_t phys = 0;
      for (auto &f : spill_files) { struct stat st; if (stat(f.c_str(), &st) == 0) phys += st.st_size; }
      counters["OUTPUT_BYTES_PHYSICAL"] += phys;
      return;
    }
    mkdirs(final_dir());
    final_out = final_dir() + "/file.out";
    final_index = final_out + ".index";
    if (num_spills == 1) {
      // sameVolRename (:730-756)
      RT_CHECK(::rename(spill_files[0].c_str(), final_out.c_str()) == 0, TEZGPU_E_IO, "rename " + spill_files[0]);
      RT_CHECK(::rename(spill_index_files[0].c_str(), final_index.c_str()) == 0, TEZGPU_E_IO, "rename " + spill_index_files[0]);
      ::rmdir(spill_dir(0).c_str());
      final_idx = spill_index[0];
      counters["SHUFFLE_CHUNK_COUNT"] = 1;
      struct stat st;
      stat(final_out.c_str(), &st);
      counters["OUTPUT_BYTES_PHYSICAL"] += st.st_size;
      return;
    }
    // final merge across spills, every partition at once on the device (:774-836)
    std::vector<std::vector<uint8_t>> bytes(num_spills);
    std::vector<tezgpu_segment> segs;
    for (int s = 0; s < num_spills; s++) {
      bytes[s] = read_file(spill_files[s]);
      counters["ADDITIONAL_SPILLS_BYTES_READ"] += (int64_t)bytes[s].size();
      for (int p = 0; p < P; p++) {
        int64_t start = spill_index[s][3 * p], raw = spill_index[s][3 * p + 1], part_len = spill_index[s][3 * p + 2];
        if (raw > 6 || (!gc.send_empty_partition_details && part_len > 0)) {  // TezIndexRecord.hasData (:51-55)
          tezgpu_segment sg;
          sg.data = bytes[s].data() + start;
          sg.len = (uint64_t)part_len;
          sg.flags = TEZGPU_SEG_HAS_HEADER;
          sg.partition = (uint32_t)p;
          segs.push_back(sg);
        }
      }
    }
    tezgpu_conf mc = gc;
    mc.fixed_key_len = mc.fixed_val_len = 0;
    tezgpu_merger *m = nullptr;
    gpu_check(tezgpu_merge_open(&mc, segs.data(), (uint32_t)segs.size(), &m));
    final_idx.assign((size_t)P * 3, 0);
    tezgpu_stats st;
    // TezMerger.merge(..., checkForSameKeys = merger.needsRLE()) into Writer(..., rle = merger.needsRLE()), `merger`
    // being the SpanMerger of the last spill (SORT/PipelinedSorter.java:797-814)
    int32_t rc = tezgpu_merge_set_check_for_same_keys(m, last_spill_rle);
    // the combiner runs in the final merge once numSpills >= tez.runtime.combine.min.spills (:815-820)
    const bool combine = combine_kind != TEZGPU_COMBINE_NONE && num_spills >= min_spills_for_combine;
    if (rc == 0 && combine) rc = tezgpu_merge_set_combiner(m, combine_kind);
    if (rc == 0)
      rc = tezgpu_merge_write_partitions(m, final_out.c_str(), final_index.c_str(), /*rle=*/last_spill_rle, final_idx.data(), &st);
    uint64_t cin = 0, cout = 0;
    if (rc == 0 && combine) rc = tezgpu_merge_combine_info(m, &cin, &cout, nullptr);
    tezgpu_merge_close(m);
    gpu_check(rc);
    if (combine) count_combine(cin, cout);
    const uint64_t len = (uint64_t)st.file_out_bytes;
    counters["SPILLED_RECORDS"] += st.spilled_records;
    int64_t raw = 0;
    for (int p = 0; p < P; p++) raw += final_idx[3 * p + 1];
    counters["OUTPUT_BYTES_WITH_OVERHEAD"] += raw;
    counters["SHUFFLE_CHUNK_COUNT"] = 1;
    counters["OUTPUT_BYTES_PHYSICAL"] += (int64_t)len;
    for (int s = 0; s < num_spills; s++) {
      ::unlink(spill_files[s].c_str());
      ::unlink(spill_index_files[s].c_str());
      ::rmdir(spill_dir(s).c_str());
    }
  }
};

struct Output {
  Configuration conf;
  std::string work_dir, uid, dest_vertex, host;
  int port, P, device;
  int64_t task_memory, requested = 0, granted = -1;
  bool initialized = false, started = false, closed = false;
  bool send_empty = true, final_merge = true;
  std::map<std::string, int64_t> counters;
  GpuSorter *sorter = nullptr;
  std::vector<Event> events;
  Output(const char *c, const char *wd, const char *u, const char *dv, const char *h, int pt, int64_t mem, int p, int dev)
      : conf(c), work_dir(wd ? wd : "."), uid(u ? u : "attempt"), dest_vertex(dv ? dv : ""), host(h ? h : "localhost"),
        port(pt), P(p), device(dev), task_memory(mem) {}
  ~Output() { delete sorter; }

  void initialize() {
    // ExternalSorter.getInitialMemoryRequirement (SORT/ExternalSorter.java:330-347)
    long mb = conf.getInt(K_SORT_MB, 100);
    int64_t req = (int64_t)mb << 20;
    RT_CHECK(mb > 0 && req < task_memory, TEZGPU_E_INVALID,
             std::string(K_SORT_MB) + " " + std::to_string(mb) + " should be larger than 0 and should be less than the available task memory (MB):" +
                 std::to_string(task_memory >> 20));
    requested = req;
    send_empty = conf.getBoolean(K_EMPTY_PARTITIONS, true);
    final_merge = conf.getBoolean(K_FINAL_MERGE, true);
    initialized = true;
  }
  void start() {
    RT_CHECK(initialized, TEZGPU_E_STATE, "start() before initialize()");
    if (started) return;
    RT_CHECK(granted >= 0, TEZGPU_E_STATE, "memory update not received (MemoryUpdateCallbackHandler.validateUpdateReceived)");
    std::string sc = conf.get(K_SORTER_CLASS, "PIPELINED");
    std::transform(sc.begin(), sc.end(), sc.begin(), ::toupper);
    RT_CHECK(sc == "PIPELINED" || sc == "LEGACY", TEZGPU_E_INVALID,
             "Invalid sorter class specified in config, propertyName=" + std::string(K_SORTER_CLASS) + ", value=" + sc + ", validValues=[LEGACY, PIPELINED]");
    RT_CHECK(!conf.getBoolean(K_COMPRESS, false), TEZGPU_E_UNSUPPORTED, "tez.runtime.compress=true: IFile codecs are not supported on the device path yet");
    const int combiner = combiner_for(conf);
    const long min_spills = conf.getInt(K_COMBINE_MIN_SPILLS, 3);
    tezgpu_conf gc;
    memset(&gc, 0, sizeof(gc));
    gc.abi_version = TEZGPU_ABI_VERSION;
    gc.device = device;
    gc.num_partitions = P;
    gc.comparator = comparator_for(conf);
    std::string pc = conf.get(K_PARTITIONER, "org.apache.tez.runtime.library.partitioner.HashPartitioner");
    gc.partitioner = ends_with(pc, "HashPartitioner") ? TEZGPU_PART_HASH : TEZGPU_PART_GIVEN;
    gc.rle_policy = TEZGPU_RLE_AUTO;
    gc.send_empty_partition_details = send_empty ? 1 : 0;
    gc.sorter_impl = sc == "LEGACY" ? 1 : 0;
    gc.mem_budget_bytes = (uint64_t)granted;
    sorter = new GpuSorter(gc, granted > 0 ? granted : requested, final_merge, work_dir, uid, counters, combiner, min_spills);
    started = true;
  }
  void write(const uint8_t *k, uint32_t kl, const uint8_t *v, uint32_t vl, int32_t partition) {
    RT_CHECK(started && !closed, TEZGPU_E_STATE, "write() outside start()..close()");
    RT_CHECK(partition >= 0 || sorter->gc.partitioner == TEZGPU_PART_HASH, TEZGPU_E_UNSUPPORTED,
             "custom partitioner: the caller must pass Partitioner.getPartition(key, value, numPartitions)");
    sorter->write(k, kl, v, vl, partition);
  }

  // ShuffleUtils.generateEventOnSpill / generateDMEPayload / generateVMEvent (RL/common/shuffle/ShuffleUtils.java:288-484)
  void generate_events(const std::vector<int64_t> &idx, const std::string &path_component, int spill_id, bool last) {
    // VertexManagerEvent
    if (final_merge || last) {
      std::string vm;
      pb_int(vm, 1, counters["OUTPUT_BYTES"]);
      std::string mode = conf.get(K_REPORT_STATS, "memory_optimized");
      std::vector<int64_t> sizes(P);
      // without the final merge the event of the last spill reports the sizes accumulated over every spill
      // (partitionStats, SORT/PipelinedSorter.java:631-633 -> ExternalSorter.getPartitionStats)
      for (int p = 0; p < P; p++)
        sizes[p] = (!final_merge && sorter && (int)sorter->partition_stats.size() == P) ? sorter->partition_stats[p] : idx[3 * p + 1];
      if (mode == "precise") {
        std::string d, packed;
        for (int p = 0; p < P; p++) pb_varint(packed, (uint64_t)((sizes[p] + (1 << 20) - 1) >> 20));
        pb_bytes(d, 1, packed);
        pb_bytes(vm, 3, d);
      } else if (mode != "none" && mode != "false") {
        // DATA_RANGE_IN_MB buckets THOUSAND,HUNDRED,TEN,ONE,ZERO -> RoaringBitmap (RL/utils/DATA_RANGE_IN_MB.java:22-47)
        static const int64_t lim[5] = {1000, 100, 10, 1, 0};
        std::vector<uint32_t> vals;
        for (int p = 0; p < P; p++) {
          int64_t mbs = (sizes[p] + (1 << 20) - 1) >> 20;
          int b = 4;
          for (int r = 0; r < 5; r++) if (mbs >= lim[r]) { b = r; break; }
          vals.push_back((uint32_t)(p * 5 + b));
        }
        std::vector<uint8_t> ser = roaring_serialize(vals);
        size_t cap = 32;  // DataOutputBuffer.getData(): the whole backing array goes through the deflater
        while (cap < ser.size()) cap <<= 1;
        ser.resize(cap, 0);
        pb_bytes(vm, 2, deflate_raw(ser));
      }
      pb_int(vm, 4, counters["OUTPUT_RECORDS"]);
      Event e;
      e.type = TEZRT_EVENT_VERTEX_MANAGER;
      e.payload = vm;
      events.push_back(e);
    }
    // CompositeDataMovementEvent(0, P, DataMovementEventPayloadProto)
    std::string dm;
    bool output_generated = true;
    if (send_empty) {
      int empty = 0, highest = -1;
      for (int p = 0; p < P; p++) if (!(idx[3 * p + 1] > 6)) { empty++; highest = p; }
      output_generated = empty != P;
      if (empty > 0) {
        std::vector<uint8_t> bits((size_t)(highest + 1 + 7) / 8, 0);  // TezUtilsInternal.toByteArray(BitSet) (big-endian byte order)
        for (int p = 0; p <= highest; p++) if (!(idx[3 * p + 1] > 6)) bits[bits.size() - (size_t)p / 8 - 1] |= (uint8_t)(1u << (p % 8));
        pb_bytes(dm, 1, deflate_raw(bits));
      }
    }
    if (!send_empty || output_generated) {
      pb_bytes(dm, 2, host);
      pb_int(dm, 3, port);
      pb_bytes(dm, 4, path_component);
    }
    pb_int(dm, 5, 0);  // run_duration
    if (!final_merge) { pb_int(dm, 8, last ? 1 : 0); pb_int(dm, 9, spill_id); }
    Event e;
    e.type = TEZRT_EVENT_COMPOSITE_DATA_MOVEMENT;
    e.payload = dm;
    e.source_index_start = 0;
    e.count = P;
    events.push_back(e);
  }

  void close() {
    RT_CHECK(started, TEZGPU_E_STATE, "close() before start()");
    if (closed) return;
    sorter->flush();
    if (final_merge) generate_events(sorter->final_idx, uid, -1, true);
    else
      for (int s = 0; s < sorter->num_spills; s++)
        generate_events(sorter->spill_index[s], uid + "_" + std::to_string(s), s, s == sorter->num_spills - 1);
    closed = true;
  }
};

// ================================================================================================ input side
struct Input {
  Configuration conf;
  std::string work_dir, uid;
  int N, device;
  int64_t task_memory, requested = 0;
  bool initialized = false, started = false, ready = false;
  std::map<std::string, int64_t> counters;
  std::vector<std::vector<uint8_t>> seg_bytes;
  // per source: spill ids seen and the id carried by the event with last_event_flag (pipelined shuffle; the reference's
  // ShuffleScheduler tracks the same per input identifier: eventsProcessed / finalEventId, OG/ShuffleScheduler.java:540-600); spill id -1 = the single
  // event of a producer that ran its final merge
  struct SourceState { std::vector<int> spills; int last_id = -2; bool complete = false; };
  std::vector<SourceState> delivered;
  int num_delivered = 0;
  tezgpu_merger *merger = nullptr;
  int cmp = 0;
  // iterator state (RL/common/ValuesIterator.java:91-201)
  std::vector<uint8_t> batch, next_batch_buf;
  std::vector<tezgpu_kv_index> idx;
  uint32_t bn = 0, bi = 0;
  std::vector<uint8_t> cur_key;
  bool have_rec = false, eos = false, in_group = false, first_of_group = false;

  Input(const char *c, const char *wd, const char *u, int64_t mem, int n, int dev)
      : conf(c), work_dir(wd ? wd : "."), uid(u ? u : "attempt"), N(n), device(dev), task_memory(mem), delivered(n) {}
  ~Input() { if (merger) tezgpu_merge_close(merger); }

  void initialize() {
    // OrderedGroupedKVInput.initialize (:100-125): Shuffle memory = shuffle.fetch.buffer.percent of the task memory
    double pct = conf.getFloat("tez.runtime.shuffle.fetch.buffer.percent", 0.9);
    requested = (int64_t)(pct * (double)task_memory);
    cmp = comparator_for(conf);
    initialized = true;
  }
  void start() {
    RT_CHECK(initialized, TEZGPU_E_STATE, "start() before initialize()");
    started = true;
    if (N == 0) ready = true;
  }
  void add_local(int src, const char *file_out, const char *index_file, int partition, bool empty, int spill_id, bool last_event) {
    RT_CHECK(started, TEZGPU_E_STATE, "handleEvents() before start()");
    RT_CHECK(src >= 0 && src < N, TEZGPU_E_INVALID, "source index out of range");
    RT_CHECK(spill_id >= -1, TEZGPU_E_INVALID, "bad spill id");
    SourceState &ss = delivered[src];
    if (spill_id < 0) {
      if (ss.complete) return;  // duplicate event for an already fetched input
      RT_CHECK(ss.spills.empty(), TEZGPU_E_STATE, "final-merge event for a source that already delivered spill events");
      ss.complete = true;
    } else {
      RT_CHECK(!(ss.complete && ss.last_id == -2), TEZGPU_E_STATE, "spill event for a source that already delivered its final output");
      for (int id : ss.spills) if (id == spill_id) return;  // duplicate spill event
      RT_CHECK(ss.last_id == -2 || spill_id < ss.last_id, TEZGPU_E_INVALID, "spill id beyond the one flagged as last");
      ss.spills.push_back(spill_id);
      if (last_event) {
        for (int id : ss.spills) RT_CHECK(id <= spill_id, TEZGPU_E_INVALID, "spill id beyond the one flagged as last");
        ss.last_id = spill_id;
      }
      ss.complete = ss.last_id >= 0 && (int)ss.spills.size() == ss.last_id + 1;
    }
    if (ss.complete) num_delivered++;
    if (empty) { counters["NUM_SKIPPED_INPUTS"]++; return; }
    // TezSpillRecord(indexFile): P x 3 big-endian longs + checksum (SORT/TezSpillRecord.java:76-109)
    std::vector<uint8_t> ib = read_file(index_file);
    RT_CHECK(ib.size() >= 8 && (ib.size() - 8) % 24 == 0, TEZGPU_E_FORMAT, std::string("bad index file ") + index_file);
    int P = (int)((ib.size() - 8) / 24);
    RT_CHECK(partition >= 0 && partition < P, TEZGPU_E_INVALID, "partition outside the producer's index");
    uLong crc = crc32(0L, Z_NULL, 0);
    crc = crc32(crc, ib.data(), (uInt)(ib.size() - 8));
    uint64_t stored = 0;
    for (int b = 0; b < 8; b++) stored = (stored << 8) | ib[ib.size() - 8 + b];
    RT_CHECK(stored == (uint64_t)crc, TEZGPU_E_FORMAT, std::string("Checksum error reading spill index: ") + index_file);
    auto be64 = [&](size_t o) { uint64_t v = 0; for (int b = 0; b < 8; b++) v = (v << 8) | ib[o + b]; return (int64_t)v; };
    int64_t start = be64((size_t)partition * 24), raw = be64((size_t)partition * 24 + 8), part = be64((size_t)partition * 24 + 16);
    if (!(raw > 6)) { counters["NUM_SKIPPED_INPUTS"]++; return; }  // !hasData
    seg_bytes.push_back(read_file(file_out, (uint64_t)start, part));
    counters["NUM_SHUFFLED_INPUTS"]++;
    counters["SHUFFLE_BYTES"] += part;
    counters["SHUFFLE_BYTES_DECOMPRESSED"] += raw;
    counters["SHUFFLE_BYTES_DISK_DIRECT"] += part;
  }
  void wait_ready() {
    RT_CHECK(started, TEZGPU_E_STATE, "waitForInputReady() before start()");
    RT_CHECK(num_delivered == N, TEZGPU_E_STATE,
             "waitForInputReady(): " + std::to_string(N - num_delivered) + " physical inputs have not been delivered");
    if (ready) return;
    tezgpu_conf gc;
    memset(&gc, 0, sizeof(gc));
    gc.abi_version = TEZGPU_ABI_VERSION;
    gc.device = device;
    gc.num_partitions = 1;
    gc.comparator = cmp;
    gc.partitioner = TEZGPU_PART_GIVEN;
    std::vector<tezgpu_segment> segs(seg_bytes.size());
    for (size_t i = 0; i < seg_bytes.size(); i++) {
      segs[i].data = seg_bytes[i].data();
      segs[i].len = seg_bytes[i].size();
      segs[i].flags = TEZGPU_SEG_HAS_HEADER;
      segs[i].partition = 0;
    }
    gpu_check(tezgpu_merge_open(&gc, segs.data(), (uint32_t)segs.size(), &merger));  // MergeManager.finalMerge -> TezMerger.merge
    counters["MERGED_MAP_OUTPUTS"] += (int64_t)segs.size();
    seg_bytes.clear();
    batch.resize(8u << 20);
    idx.resize(1u << 16);
    ready = true;
  }
  bool fetch() {  // next record of the merged stream into (idx[bi])
    if (eos) return false;
    if (bi + 1 < bn) { bi++; return true; }
    uint32_t n = 0;
    gpu_check(tezgpu_merge_next_batch(merger, batch.data(), batch.size(), idx.data(), (uint32_t)idx.size(), &n));
    if (n == 0) { eos = true; return false; }
    bn = n;
    bi = 0;
    return true;
  }
  // KeyValuesReader.next(): ValuesIterator.moveToNext (:91-105) -- skip what is left of the current group
  bool next(const uint8_t **key, uint32_t *klen) {
    RT_CHECK(ready, TEZGPU_E_STATE, "getReader() before waitForInputReady()");
    if (!merger) return false;
    if (in_group) { const uint8_t *v; uint32_t vl; while (next_value(&v, &vl)) {} }
    if (!have_rec) { if (!fetch()) return false; have_rec = true; }
    const tezgpu_kv_index &e = idx[bi];
    cur_key.assign(batch.data() + e.key_off, batch.data() + e.key_off + e.key_len);
    in_group = true;
    first_of_group = true;
    counters["REDUCE_INPUT_GROUPS"]++;
    *key = cur_key.data();
    *klen = (uint32_t)cur_key.size();
    return true;
  }
  bool next_value(const uint8_t **val, uint32_t *vlen) {
    if (!in_group) return false;
    if (!first_of_group) {
      // readNextKey (:177-201): same group when the merger says isSameKey(), else compare the raw key bytes
      // (equal keys of the supported classes have equal serialized bytes)
      if (!fetch()) { have_rec = false; in_group = false; return false; }
      const tezgpu_kv_index &e = idx[bi];
      bool same = e.same_key || (e.key_len == cur_key.size() && memcmp(batch.data() + e.key_off, cur_key.data(), e.key_len) == 0);
      if (!same) { in_group = false; have_rec = true; return false; }
    }
    first_of_group = false;
    const tezgpu_kv_index &e = idx[bi];
    *val = batch.data() + e.val_off;
    *vlen = e.val_len;
    counters["REDUCE_INPUT_RECORDS"]++;
    return true;
  }
};

}  // namespace tezrt

using namespace tezrt;

struct tezrt_output { Output o; tezrt_output(const char *c, const char *wd, const char *u, const char *dv, const char *h, int pt, int64_t mem, int p, int dev) : o(c, wd, u, dv, h, pt, mem, p, dev) {} };
struct tezrt_input { Input i; tezrt_input(const char *c, const char *wd, const char *u, int64_t mem, int n, int dev) : i(c, wd, u, mem, n, dev) {} };

#define RT_BEGIN try {
#define RT_END } catch (const Err &e) { g_err = e.what(); return e.code; } catch (const std::exception &e) { g_err = e.what(); return TEZGPU_E_INVALID; } return 0;

extern "C" {
const char *tezrt_last_error(void) { return g_err.c_str(); }

int32_t tezrt_output_create(const char *conf, const char *work_dir, const char *unique_id, const char *dest_vertex, const char *host,
                            int32_t port, int64_t task_memory, int32_t P, int32_t device, tezrt_output **out) {
  RT_BEGIN
  RT_CHECK(out && P >= 1, TEZGPU_E_INVALID, "bad arguments");
  *out = new tezrt_output(conf, work_dir, unique_id, dest_vertex, host, port, task_memory, P, device);
  RT_END
}
int32_t tezrt_output_initialize(tezrt_output *o, int64_t *requested) { RT_BEGIN o->o.initialize(); if (requested) *requested = o->o.requested; RT_END }
int32_t tezrt_output_memory_assigned(tezrt_output *o, int64_t granted) { RT_BEGIN o->o.granted = granted; RT_END }
int32_t tezrt_output_start(tezrt_output *o) { RT_BEGIN o->o.start(); RT_END }
int32_t tezrt_output_write(tezrt_output *o, const uint8_t *k, uint32_t kl, const uint8_t *v, uint32_t vl, int32_t partition) {
  RT_BEGIN o->o.write(k, kl, v, vl, partition); RT_END
}
int32_t tezrt_output_close(tezrt_output *o, int32_t *n) { RT_BEGIN o->o.close(); if (n) *n = (int32_t)o->o.events.size(); RT_END }
int32_t tezrt_output_event(tezrt_output *o, int32_t i, int32_t *type, const uint8_t **payload, uint64_t *len, int32_t *start, int32_t *count) {
  RT_BEGIN
  RT_CHECK(i >= 0 && i < (int)o->o.events.size(), TEZGPU_E_INVALID, "event index");
  const Event &e = o->o.events[i];
  if (type) *type = e.type;
  if (payload) *payload = (const uint8_t *)e.payload.data();
  if (len) *len = e.payload.size();
  if (start) *start = e.source_index_start;
  if (count) *count = e.count;
  RT_END
}
int64_t tezrt_output_counter(tezrt_output *o, const char *name) { auto it = o->o.counters.find(name); return it == o->o.counters.end() ? 0 : it->second; }
int32_t tezrt_output_num_spills(tezrt_output *o) { return o->o.sorter ? o->o.sorter->num_spills : 0; }
const char *tezrt_output_file(tezrt_output *o) { return o->o.sorter ? o->o.sorter->final_out.c_str() : ""; }
const char *tezrt_output_index_file(tezrt_output *o) { return o->o.sorter ? o->o.sorter->final_index.c_str() : ""; }
int32_t tezrt_output_destroy(tezrt_output *o) { delete o; return 0; }

int32_t tezrt_input_create(const char *conf, const char *work_dir, const char *unique_id, int64_t task_memory, int32_t n, int32_t device,
                           tezrt_input **out) {
  RT_BEGIN
  RT_CHECK(out && n >= 0, TEZGPU_E_INVALID, "bad arguments");
  *out = new tezrt_input(conf, work_dir, unique_id, task_memory, n, device);
  RT_END
}
int32_t tezrt_input_initialize(tezrt_input *in, int64_t *requested) { RT_BEGIN in->i.initialize(); if (requested) *requested = in->i.requested; RT_END }
int32_t tezrt_input_start(tezrt_input *in) { RT_BEGIN in->i.start(); RT_END }
int32_t tezrt_input_add_local_output(tezrt_input *in, int32_t src, const char *file_out, const char *index_file, int32_t partition, int32_t empty) {
  RT_BEGIN in->i.add_local(src, file_out, index_file, partition, empty != 0, -1, true); RT_END
}
int32_t tezrt_input_add_local_spill(tezrt_input *in, int32_t src, const char *file_out, const char *index_file, int32_t partition, int32_t empty,
                                    int32_t spill_id, int32_t last_event) {
  RT_BEGIN in->i.add_local(src, file_out, index_file, partition, empty != 0, spill_id, last_event != 0); RT_END
}
int32_t tezrt_input_wait_ready(tezrt_input *in) { RT_BEGIN in->i.wait_ready(); RT_END }
int32_t tezrt_input_next(tezrt_input *in, const uint8_t **key, uint32_t *klen) {
  try { return in->i.next(key, klen) ? 1 : 0; } catch (const Err &e) { g_err = e.what(); return e.code; }
}
int32_t tezrt_input_next_value(tezrt_input *in, const uint8_t **val, uint32_t *vlen) {
  try { return in->i.next_value(val, vlen) ? 1 : 0; } catch (const Err &e) { g_err = e.what(); return e.code; }
}
int64_t tezrt_input_counter(tezrt_input *in, const char *name) { auto it = in->i.counters.find(name); return it == in->i.counters.end() ? 0 : it->second; }
int32_t tezrt_input_destroy(tezrt_input *in) { delete in; return 0; }
}
