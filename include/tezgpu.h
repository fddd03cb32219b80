/*
 * tezgpu.h -- C ABI of libtezgpu.so: B200-native (sm_100a) replacement of the Tez shuffle sort/merge hot path.
 *
 * This is the drop-in boundary (SURVEY.md 8b).  Plain pointers and sizes only -- no torch / C++ types.
 * Each entry point names the reference interface it replaces.  Paths are relative to
 * /root/reference/tez-runtime-library/src/main/java/org/apache/tez/runtime/library/ (RL/), SORT/ = RL/common/sort/impl/.
 *
 * Conventions
 *   - every function returns int32: 0 = ok, <0 = TEZGPU_E_*; tezgpu_last_error() gives the message of the last
 *     failure on the calling thread (the JNI stub turns it into java.io.IOException, like every failure of the
 *     reference path: SORT/PipelinedSorter.java:400-413).
 *   - no exceptions cross the boundary; handles are opaque; one producer thread per handle; handles independent.
 *   - the caller owns every buffer it passes, for the duration of the call only; the library owns device memory.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with TEZGPU_E_CUDA.
 */
#ifndef TEZGPU_H
#define TEZGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TEZGPU_ABI_VERSION 1

/* error codes */
#define TEZGPU_OK 0
#define TEZGPU_E_INVALID (-1)     /* bad argument / illegal partition ("Illegal partition for ...", PipelinedSorter.java:410-413) */
#define TEZGPU_E_CUDA (-2)        /* CUDA runtime failure (incl. no device) */
#define TEZGPU_E_NOMEM (-3)       /* device or host allocation failed -> task attempt fails, no CPU fallback */
#define TEZGPU_E_IO (-4)          /* file write failed */
#define TEZGPU_E_FORMAT (-5)      /* malformed IFile segment / checksum mismatch (IFileInputStream.java:235-289) */
#define TEZGPU_E_UNSUPPORTED (-6) /* comparator / partitioner / codec outside the device-supported closed set */
#define TEZGPU_E_STATE (-7)       /* call sequence violation (e.g. collect after flush) */

/* key comparator = RawComparator selected by ConfigUtils.getIntermediateOutputKeyComparator (RL/common/ConfigUtils.java:92-100) */
#define TEZGPU_CMP_BYTES 0          /* TezBytesComparator / raw bytes (RL/common/comparator/TezBytesComparator.java:37-41) */
#define TEZGPU_CMP_TEXT 1           /* hadoop Text.Comparator: skip the vint length prefix, then unsigned bytes */
#define TEZGPU_CMP_BYTESWRITABLE 2  /* hadoop BytesWritable.Comparator: skip the 4-byte length, then unsigned bytes */
#define TEZGPU_CMP_INT 3            /* IntWritable.Comparator: 4-byte big-endian signed */
#define TEZGPU_CMP_LONG 4           /* LongWritable.Comparator: 8-byte big-endian signed */

/* partitioner (RL/partitioner/HashPartitioner.java:33-35) */
#define TEZGPU_PART_GIVEN 0         /* caller computed Partitioner.getPartition in Java and passes the ids */
#define TEZGPU_PART_HASH 1          /* device computes (key.hashCode() & MAX_VALUE) % P for the comparator's key class */

/* RLE policy of IFile.Writer (SORT/IFile.java:541-544; decision SORT/PipelinedSorter.java:1436-1438) */
#define TEZGPU_RLE_AUTO (-1)        /* on iff (#adjacent equal keys in sorted order) > 0.1 * records -- see DESIGN.md "RLE decision" */
#define TEZGPU_RLE_OFF 0
#define TEZGPU_RLE_ON 1

/* sorter_impl = 2: the writer behind UnorderedPartitionedKVOutput (RL/common/writers/UnorderedPartitionedKVWriter.java):
 * records are only partitioned; every partition's segment holds its records NEWEST FIRST (the per-partition chain of
 * :459-472 walked by writePartition :688-703 -- the order the reference writes when everything fits one buffer), IFile
 * without run-length encoding (:1092), no bytes and an all-zero index entry for a partition without records (mergeAll
 * :1058-1144).  The comparator is ignored.  With several buffers / spills the reference's order inside a partition
 * depends on buffer arithmetic and thread timing: parity is then the identical index + the per-partition multiset. */
#define TEZGPU_SORTER_UNORDERED 2

/* combiner (tez.runtime.combiner.class = MRCombiner over a sum reducer; SORT/PipelinedSorter.java:601-609,815-820):
 * the sorted records of every partition are replaced by one record per group of equal keys -- the group's key and the
 * sum of its values, Java int / long wrap-around -- before they are written.  Combined keys are unique within a
 * partition, so a combined segment holds no REPEAT_KEY record. */
#define TEZGPU_COMBINE_NONE 0
#define TEZGPU_COMBINE_INT_SUM 1    /* IntSumReducer: values are 4-byte big-endian IntWritable */
#define TEZGPU_COMBINE_LONG_SUM 2   /* LongSumReducer (new and old API): values are 8-byte big-endian LongWritable */

typedef struct tezgpu_conf {
  int32_t abi_version;                  /* TEZGPU_ABI_VERSION */
  int32_t device;                       /* CUDA ordinal */
  int32_t num_partitions;               /* numPhysicalOutputs (RL/output/OrderedPartitionedKVOutput.java:91-110) */
  int32_t comparator;                   /* TEZGPU_CMP_* */
  int32_t partitioner;                  /* TEZGPU_PART_* */
  int32_t rle_policy;                   /* TEZGPU_RLE_* */
  int32_t send_empty_partition_details; /* tez.runtime.empty.partitions.info-via-events.enabled (default 1) */
  int32_t sorter_impl;                  /* 0 = PipelinedSorter (default), 1 = DefaultSorter ("LEGACY"): only changes the AUTO RLE rule,
                                           2 = TEZGPU_SORTER_UNORDERED: UnorderedPartitionedKVWriter (partition only, no key order) */
  uint32_t fixed_key_len;               /* >0 with fixed_val_len: records are packed key||value of constant width */
  uint32_t fixed_val_len;
  uint64_t mem_budget_bytes;            /* granted by OutputContext.requestInitialMemory; 0 = no limit.  Enforced on the key+value
                                           bytes collected since the last reset: a collect that would pass it fails with
                                           TEZGPU_E_NOMEM and the caller spills (flush + reset), like PipelinedSorter when its
                                           kvbuffer is full (SORT/PipelinedSorter.java:415-444) */
} tezgpu_conf;

/* counters + per-partition results; mirrors TezSpillRecord / TezIndexRecord and the ExternalSorter counters
 * (SORT/TezSpillRecord.java:48-52, SORT/ExternalSorter.java:141-167) */
typedef struct tezgpu_stats {
  int64_t output_records;               /* OUTPUT_RECORDS */
  int64_t output_bytes;                 /* OUTPUT_BYTES: sum(keyLen+valLen) */
  int64_t output_bytes_with_overhead;   /* OUTPUT_BYTES_WITH_OVERHEAD: sum(rawLength) */
  int64_t output_bytes_physical;        /* OUTPUT_BYTES_PHYSICAL: file.out length */
  int64_t spilled_records;              /* SPILLED_RECORDS */
  int64_t file_out_bytes;               /* bytes produced for file.out */
  int32_t num_spills;                   /* always 1: HBM is the sort buffer (PipelinedSorter.flush numSpills==1 branch :730-756) */
  int32_t rle_used;
  int64_t adjacent_equal_keys;
  int64_t tie_records;                  /* records that needed key-suffix refinement after the prefix radix sort */
  float ms_stage, ms_sort, ms_ties, ms_emit, ms_total; /* device times of the last flush (CUDA events) */
  int32_t kernel_launches;              /* kernels launched by the last flush / merge */
  float ms_emit_kernel;                 /* device time of the gather+emit kernel alone (CUDA events around its launch) */
} tezgpu_stats;

typedef struct tezgpu_sorter tezgpu_sorter;
typedef struct tezgpu_merger tezgpu_merger;

const char *tezgpu_last_error(void);
int32_t tezgpu_abi_version(void);
/* number of visible CUDA devices (0 when none; never falls back to CPU) */
int32_t tezgpu_device_count(void);

/* ------------------------------------------------------------------------------------------------------------------
 * Sorter: replaces PipelinedSorter / DefaultSorter behind ExternalSorter (SORT/ExternalSorter.java:74-92,281-288)
 * ---------------------------------------------------------------------------------------------------------------- */

/* replaces `new PipelinedSorter(outputContext, conf, numOutputs, initialMemory)` (RL/output/OrderedPartitionedKVOutput.java:116-160) */
int32_t tezgpu_sorter_create(const tezgpu_conf *conf, tezgpu_sorter **out);

/* replaces PipelinedSorter.write/collect (SORT/PipelinedSorter.java:387-466), batched: one JNI crossing per n records.
 * kv holds the serialized records; record i's key is kv[key_off[i] .. val_off[i]) and its value kv[val_off[i] .. +val_len[i])
 * (the {KEYSTART, VALSTART, VALLEN} metadata triple of :459-462).  partition may be NULL when conf.partitioner==HASH.
 * Bytes are copied before the call returns (the caller reuses its buffers, WordCount.java:74-75,95-97). */
int32_t tezgpu_sorter_collect_batch(tezgpu_sorter *h, const uint8_t *kv, uint64_t kv_bytes, const uint32_t *key_off,
                                    const uint32_t *val_off, const uint32_t *val_len, const int32_t *partition,
                                    uint32_t n);

/* fixed-width fast path of the above: n records of (fixed_key_len + fixed_val_len) bytes packed back to back */
int32_t tezgpu_sorter_collect_fixed(tezgpu_sorter *h, const uint8_t *kv, const int32_t *partition, uint64_t n);

/* replaces PipelinedSorter.flush()+spill() (SORT/PipelinedSorter.java:558-647,664-859): sorts by (partition, key),
 * writes file.out (concatenated IFile segments, mode 0640) and file.out.index (TezSpillRecord), fills stats and
 * index[3*P] = (startOffset, rawLength, partLength) per partition.  index may be NULL. */
int32_t tezgpu_sorter_flush(tezgpu_sorter *h, const char *out_path, const char *index_path, int64_t *index,
                            tezgpu_stats *stats);

/* same, into caller memory instead of files (tests / in-process consumers). out_cap >= tezgpu_sorter_output_bound(h).
 * index_out (may be NULL) receives the P*24+8 bytes of file.out.index. */
int32_t tezgpu_sorter_flush_to_memory(tezgpu_sorter *h, uint8_t *out, uint64_t out_cap, uint64_t *out_len,
                                      uint8_t *index_out, int64_t *index, tezgpu_stats *stats);
uint64_t tezgpu_sorter_output_bound(const tezgpu_sorter *h);

/* replaces ExternalSorter.close() (SORT/ExternalSorter.java:281-288) */
int32_t tezgpu_sorter_destroy(tezgpu_sorter *h);
/* forgets the collected records but keeps every device / pinned allocation, so a container-reused task
 * (tez.am.container.reuse) can run its next output through the same handle */
int32_t tezgpu_sorter_reset(tezgpu_sorter *h);

/* Device-resident variant (records already in HBM; used by the multi-GPU shuffle and by bench.py's kernel-only
 * measurement).  d_kv: n packed fixed-width records on conf.device; d_partition may be 0.  d_out receives file.out
 * bytes (capacity out_cap); index (host, 3*P int64) and stats are filled after an internal stream sync.
 * Runs on the handle's stream (tezgpu_sorter_stream). */
int32_t tezgpu_sorter_sort_device_fixed(tezgpu_sorter *h, const void *d_kv, const void *d_partition, uint64_t n,
                                        void *d_out, uint64_t out_cap, uint64_t *out_len, int64_t *index,
                                        tezgpu_stats *stats);
/* cudaStream_t of the handle, as an opaque pointer (so callers can record events on it) */
void *tezgpu_sorter_stream(tezgpu_sorter *h);

/* runCombineProcessor at spill time (SORT/PipelinedSorter.java:601-609): every flush writes the combined records.
 * Call before the first collect or right after a reset; the kind stays set across resets.  TEZGPU_E_UNSUPPORTED on a
 * TEZGPU_SORTER_UNORDERED handle; TEZGPU_E_INVALID when fixed_val_len is set and is not the kind's value width.  A
 * collected value of the wrong width makes the flush fail with TEZGPU_E_INVALID.  With a combiner, stats.spilled_records
 * and output_bytes_with_overhead count the combined records, output_records / output_bytes / adjacent_equal_keys /
 * rle_used the collected ones (the RLE decision is taken before the combine). */
int32_t tezgpu_sorter_set_combiner(tezgpu_sorter *h, int32_t kind);
/* records into and out of the combine of the last flush (both 0 without a combiner) and its device time */
int32_t tezgpu_sorter_combine_info(tezgpu_sorter *h, uint64_t *records_in, uint64_t *records_out, float *ms);

/* ------------------------------------------------------------------------------------------------------------------
 * Merger: replaces TezMerger.merge(...) -> TezRawKeyValueIterator (SORT/TezMerger.java:717-912,
 * SORT/TezRawKeyValueIterator.java:33-87) as called from OG/MergeManager.java:804-811,899-903,1035-1041,1197-1199
 * and PipelinedSorter.flush :774-836.
 * ---------------------------------------------------------------------------------------------------------------- */
#define TEZGPU_SEG_HAS_HEADER 1u   /* on-disk layout: 'T','I','F',flag + body + crc  (DiskSegment); else body + crc (InMemoryReader) */
#define TEZGPU_SEG_DEVICE 2u       /* data is a device pointer on conf.device */
#define TEZGPU_SEG_VERIFIED 4u     /* the transport already verified this segment's checksum while copying it (as
                                      IFile.Reader.readToMemory does for fetched MEMORY outputs, SORT/IFile.java:764-809,
                                      whose InMemoryReader then never re-checks): tezgpu_fetch_segments_verified */

typedef struct tezgpu_segment {
  const void *data;
  uint64_t len;
  uint32_t flags;
  uint32_t partition;              /* output partition this segment belongs to (0 for a single-partition merge) */
} tezgpu_segment;

/* one merged record: offsets into the batch buffer returned by tezgpu_merge_next_batch */
typedef struct tezgpu_kv_index {
  uint32_t key_off, key_len, val_off, val_len;
  uint32_t same_key;               /* TezRawKeyValueIterator.isSameKey() */
} tezgpu_kv_index;

/* opens the k-way merge over nseg sorted IFile segments: verifies checksums, parses, merges on device */
int32_t tezgpu_merge_open(const tezgpu_conf *conf, const tezgpu_segment *segs, uint32_t nseg, tezgpu_merger **out);
/* runs a new merge through an existing handle, keeping its device allocations (the per-step reduce side of the
 * multi-GPU shuffle; a container-reused task) */
int32_t tezgpu_merge_reopen(tezgpu_merger *m, const tezgpu_segment *segs, uint32_t nseg);
/* MergeQueue's checkForSameKeys constructor argument (SORT/TezMerger.java:560-573; default true like the reference's
 * other constructors, :519).  When 0, isSameKey() -- and therefore REPEAT_KEY in tezgpu_merge_write_* -- is reported
 * only for records that were run-length encoded in their input segment, never across segment boundaries
 * (adjustPriorityQueue / compareKeyWithNextTopKey, :597-652).  PipelinedSorter's final merge passes
 * merger.needsRLE() here AND as the writer's rle (SORT/PipelinedSorter.java:797-814).  Call before next_batch / write. */
int32_t tezgpu_merge_set_check_for_same_keys(tezgpu_merger *m, int32_t check_for_same_keys);
/* total records / key+value bytes of the merged stream */
/* diagnostics: how the last open / reopen located the records -- mode 0: fixed framing, records addressed in place
 * (no parse); 1: parallel window parser (by_hand = windows whose guessed entry was wrong and that the chase walked
 * itself); 2: sequential walker (one lane per segment: taken when the window parser meets a malformed record) */
int32_t tezgpu_merge_parse_info(tezgpu_merger *m, int32_t *mode, int32_t *by_hand);
int32_t tezgpu_merge_counts(tezgpu_merger *m, uint64_t *records, uint64_t *kv_bytes);
/* replaces the next()/getKey()/getValue()/isSameKey() loop: fills up to idx_cap records (key||value bytes appended to
 * out_kv, at most cap bytes); *n = 0 at end of stream */
int32_t tezgpu_merge_next_batch(tezgpu_merger *m, uint8_t *out_kv, uint64_t cap, tezgpu_kv_index *idx,
                                uint32_t idx_cap, uint32_t *n);
/* replaces TezMerger.writeFile(iter, new IFile.Writer(..., rle)) (SORT/TezMerger.java:215-245): one IFile segment.
 * path may be NULL when out != NULL.  raw_len / part_len as IFile.Writer.getRawLength / getCompressedLength. */
int32_t tezgpu_merge_write_ifile(tezgpu_merger *m, const char *path, uint8_t *out, uint64_t out_cap, int32_t rle,
                                 int64_t *raw_len, int64_t *part_len, tezgpu_stats *stats);
uint64_t tezgpu_merge_output_bound(const tezgpu_merger *m);
/* device-resident output of the merged IFile segment (multi-GPU reduce side, bench) */
int32_t tezgpu_merge_write_ifile_device(tezgpu_merger *m, void *d_out, uint64_t out_cap, int32_t rle, int64_t *raw_len,
                                        int64_t *part_len, tezgpu_stats *stats);
/* Batched reduce side (multi-GPU shuffle): the merger was opened with conf.num_partitions = P and every segment
 * names its partition; writes the P merged segments back to back like a file.out and fills index[3*P]. */
int32_t tezgpu_merge_write_partitions_device(tezgpu_merger *m, void *d_out, uint64_t out_cap, int32_t rle,
                                             uint64_t *out_len, int64_t *index, tezgpu_stats *stats);
/* same, written to file.out + file.out.index (mode 0640): the final merge of PipelinedSorter.flush over several spills
 * (SORT/PipelinedSorter.java:774-836) */
int32_t tezgpu_merge_write_partitions(tezgpu_merger *m, const char *out_path, const char *index_path, int32_t rle,
                                      int64_t *index, tezgpu_stats *stats);
/* combiner of a combining merge (PipelinedSorter.flush with numSpills >= tez.runtime.combine.min.spills, :815-820;
 * MergeManager's mem->disk merges, OG/MergeManager.java:899-911): applies to the tezgpu_merge_write_* entry points;
 * tezgpu_merge_next_batch stays the uncombined TezRawKeyValueIterator stream */
int32_t tezgpu_merge_set_combiner(tezgpu_merger *m, int32_t kind);
int32_t tezgpu_merge_combine_info(tezgpu_merger *m, uint64_t *records_in, uint64_t *records_out, float *ms);
void *tezgpu_merge_stream(tezgpu_merger *m);
int32_t tezgpu_merge_close(tezgpu_merger *m);

/* ---------------------------------------------------------------------------------------------------------------
 * Shuffle transfer between the GPUs of one box (NVLink / NVSwitch).
 * Replaces the ShuffleHandler HTTP GET + FetcherOrderedGrouped.copyMapOutput round trip
 * (OG/FetcherOrderedGrouped.java:437-632, OG/ShuffleScheduler.java:1370-1470): the producer keeps file.out in an
 * exportable device buffer, the consumer maps it (CUDA IPC) and pulls the byte ranges of its partitions with one
 * kernel running on every SM.  Handles are 64 opaque bytes the host layer ships with the DataMovementEvent.
 * --------------------------------------------------------------------------------------------------------------- */
#define TEZGPU_PEER_HANDLE_BYTES 64
/* device buffer another process on the same box may map; *handle_out receives the 64-byte export handle */
int32_t tezgpu_peer_alloc(int32_t device, uint64_t bytes, void **dptr, uint8_t *handle_out);
int32_t tezgpu_peer_free(int32_t device, void *dptr);
/* maps a buffer exported by another process (any device of the box) into this process; enables peer access */
int32_t tezgpu_peer_open(int32_t device, const uint8_t *handle, void **dptr);
int32_t tezgpu_peer_close(int32_t device, void *dptr);
typedef struct tezgpu_copy_range {
  const void *src;                 /* device address (local, or a peer mapping from tezgpu_peer_open) */
  void *dst;                       /* device address on `device`; fastest when (dst - src) is a multiple of 16 */
  uint64_t len;
} tezgpu_copy_range;
/* copies n ranges with one launch on `stream` (a cudaStream_t, NULL = the legacy default stream) and returns once
 * the bytes have landed */
int32_t tezgpu_fetch_ranges(int32_t device, const tezgpu_copy_range *ranges, uint32_t n, void *stream,
                            float *ms_kernel);

/* The same pull with every segment's IFile checksum verified on the bytes as they pass through the copy kernel -- what
 * IFile.Reader.readToMemory does when FetcherOrderedGrouped fetches a map output to MEMORY (SORT/IFile.java:764-809,
 * OG/FetcherOrderedGrouped.java:519-533).  One entry per (non-empty) segment; src may be a peer mapping, dst is local,
 * (dst - src) must be a multiple of 16 and only the bytes of the listed segments move.  Fails with TEZGPU_E_FORMAT
 * ("IFile checksum mismatch in fetched segment i") like the reference's ChecksumException; segments that passed may be
 * handed to tezgpu_merge_open with TEZGPU_SEG_VERIFIED so the merge does not read them a second time to check. */
typedef struct tezgpu_fetch_segment {
  const void *src;
  void *dst;
  uint64_t len;                    /* whole segment: header + body + 4 checksum bytes */
  uint32_t flags;                  /* TEZGPU_SEG_HAS_HEADER */
  uint32_t reserved;
} tezgpu_fetch_segment;
int32_t tezgpu_fetch_segments_verified(int32_t device, const tezgpu_fetch_segment *segs, uint32_t n, void *stream,
                                       float *ms_kernel);

/* ---- SURVEY 8 f-2: the ShuffleHandler <-> FetcherOrderedGrouped wire format, for consumers outside the NVLink domain
 * (and unmodified fetchers).  Per map output and reducer: ShuffleHeader (OG/ShuffleHeader.java:101-106:
 * Text.writeString(mapId), vlong compressedLength = partLength, vlong uncompressedLength = rawLength, vint forReduce)
 * followed by partLength bytes of the partition's IFile segment (OG/FetcherOrderedGrouped.java:437-632 reads exactly
 * that).  Host-side framing; the segment bytes are copied out of the device-resident file.out. */
uint64_t tezgpu_shuffle_header_size(const char *map_id, int64_t part_len, int64_t raw_len, int32_t reduce);
int32_t tezgpu_shuffle_header_write(const char *map_id, int64_t part_len, int64_t raw_len, int32_t reduce, uint8_t *out,
                                    uint64_t cap, uint64_t *len);
/* ShuffleHeader.readFields (:82-87, map id at most 1000 bytes); consumed = header bytes */
int32_t tezgpu_shuffle_header_read(const uint8_t *in, uint64_t avail, char *map_id, uint64_t map_id_cap, int64_t *part_len,
                                   int64_t *raw_len, int32_t *reduce, uint64_t *consumed);
/* response body for reducers [reduce0, reduce0 + nreduce) of ONE map output whose file.out lives in device memory:
 * index = the 3 * P int64 triples (start, rawLength, partLength) of its spill record; out = host (ideally pinned) buffer
 * of at least tezgpu_shuffle_serve_bound bytes; returns after the copies completed */
uint64_t tezgpu_shuffle_serve_bound(const char *map_id, const int64_t *index, int32_t reduce0, int32_t nreduce);
int32_t tezgpu_shuffle_serve(int32_t device, const void *d_file_out, const int64_t *index, const char *map_id,
                             int32_t reduce0, int32_t nreduce, uint8_t *out, uint64_t cap, uint64_t *len, void *stream);
/* consumer side: splits a response body into its segments (what copyMapOutput does header by header); every segment is
 * in[offset .. offset + part_len) and can go to tezgpu_merge_open as a host segment with TEZGPU_SEG_HAS_HEADER */
typedef struct tezgpu_wire_segment {
  char map_id[1008];
  int64_t part_len;
  int64_t raw_len;
  uint64_t offset;
  int32_t reduce;
  int32_t reserved;
} tezgpu_wire_segment;
int32_t tezgpu_shuffle_receive(const uint8_t *in, uint64_t len, tezgpu_wire_segment *segs, uint32_t cap, uint32_t *n);

/* diagnostics: host-side emulation of the device's tiled CRC algebra (same tables, no GPU needed) */
uint32_t tezgpu_debug_crc_emulate(const uint8_t *body, uint64_t len, uint32_t piece_bytes, uint32_t lead);

/* diagnostics: host-side run of the TMA emit kernel's chunk assembly (same template code, no GPU needed) */
uint32_t tezgpu_debug_assemble_emulate(const uint8_t *stage, uint32_t nr, uint32_t stride, const uint8_t *hdr,
                                       uint32_t hdr_len, uint32_t lead, int32_t first, int32_t last, uint8_t *image_out,
                                       uint32_t image_cap);

/* diagnostics: host-side run of the chunk-interleaved CRC fold of the emit / verify kernels (ilp: two-deep form) */
uint32_t tezgpu_debug_chunk_fold_emulate(const uint8_t *data, uint32_t nchunks, int32_t ilp);

uint32_t tezgpu_debug_runs_assemble_emulate(const uint8_t *staging, uint32_t staging_len, const uint32_t *src, uint32_t nr,
                                            uint32_t rec_size, uint32_t lead, int32_t first, int32_t last,
                                            uint8_t *image_out, uint32_t image_cap);

#ifdef __cplusplus
}
#endif
#endif /* TEZGPU_H */
