/*
 * GpuSorter -- the ExternalSorter seam of OrderedPartitionedKVOutput backed by libtezgpu.so (include/tezgpu.h).
 *
 * Drop-in position: add `GPU` to OrderedPartitionedKVOutput.SorterImpl and construct this class where start() builds
 * PipelinedSorter / DefaultSorter (tez-runtime-library/.../output/OrderedPartitionedKVOutput.java:116-160).  Everything
 * else of the plugin -- events, counters, file names, the KeyValuesWriter -- is the reference's own code.
 *
 * NOT COMPILED IN THIS REPOSITORY: the build image has no JDK (java, javac and mvn are absent).  The C side of every
 * native method below is jni/tezgpu_jni.c; both follow include/tezgpu.h, which IS built and tested here through ctypes.
 */
package org.apache.tez.runtime.library.common.sort.impl;

import java.io.IOException;
import java.nio.ByteBuffer;
import java.nio.ByteOrder;
import java.nio.IntBuffer;

import org.apache.hadoop.conf.Configuration;
import org.apache.hadoop.io.BytesWritable;
import org.apache.hadoop.io.IntWritable;
import org.apache.hadoop.io.LongWritable;
import org.apache.hadoop.io.RawComparator;
import org.apache.hadoop.io.Text;
import org.apache.tez.common.counters.TaskCounter;
import org.apache.tez.runtime.api.OutputContext;
import org.apache.tez.runtime.library.common.ConfigUtils;
import org.apache.tez.runtime.library.common.comparator.TezBytesComparator;
import org.apache.tez.runtime.library.partitioner.HashPartitioner;

/** Replaces PipelinedSorter.collect / sort / spill / flush (PipelinedSorter.java:387-466, 558-859). */
public class GpuSorter extends ExternalSorter {
  static {
    System.loadLibrary("tezgpu_jni"); // jni/tezgpu_jni.c, linked against libtezgpu.so
  }

  // ids of include/tezgpu.h
  static final int CMP_BYTES = 0, CMP_TEXT = 1, CMP_BYTESWRITABLE = 2, CMP_INT = 3, CMP_LONG = 4;
  static final int PART_GIVEN = 0, PART_HASH = 1;
  static final int COMBINE_NONE = 0, COMBINE_INT_SUM = 1, COMBINE_LONG_SUM = 2;
  private static final int BATCH_BYTES = 32 << 20;
  private static final int BATCH_RECORDS = 1 << 20;

  private long handle; // tezgpu_sorter*
  private final ByteBuffer kv = ByteBuffer.allocateDirect(BATCH_BYTES).order(ByteOrder.nativeOrder());
  private final IntBuffer keyOff = direct(BATCH_RECORDS), valOff = direct(BATCH_RECORDS), valLen = direct(BATCH_RECORDS),
      part = direct(BATCH_RECORDS);
  private final boolean deviceHash;
  private final ByteBufferOutputStream sink = new ByteBufferOutputStream(kv);
  private int n;
  private long collectedBytes;
  private boolean lastSpillRle;
  private final int combineKind;
  private final int minSpillsForCombine;

  private static IntBuffer direct(int ints) {
    return ByteBuffer.allocateDirect(4 * ints).order(ByteOrder.nativeOrder()).asIntBuffer();
  }

  public GpuSorter(OutputContext outputContext, Configuration conf, int numOutputs, long initialMemoryAvailable)
      throws IOException {
    super(outputContext, conf, numOutputs, initialMemoryAvailable);
    deviceHash = partitioner instanceof HashPartitioner;
    handle = nativeCreate(numOutputs, comparatorId(comparator, conf), deviceHash ? PART_HASH : PART_GIVEN,
        sendEmptyPartitionDetails, initialMemoryAvailable, /* CUDA ordinal, from the container's environment */
        Integer.parseInt(System.getenv().getOrDefault("TEZGPU_DEVICE", "0")));
    keySerializer.open(sink);
    valSerializer.open(sink);
    combineKind = combinerKind(combiner, conf);
    minSpillsForCombine = conf.getInt("tez.runtime.combine.min.spills", 3);
    if (combineKind != COMBINE_NONE) nativeSetCombiner(handle, combineKind); // tezgpu_sorter_set_combiner
  }

  /**
   * The combiner ExternalSorter instantiated (TezRuntimeUtils.instantiateCombiner): MRCombiner over a sum reducer runs on
   * the device; any other combiner is not run, as before.  MRCombiner reads the reducer from mapreduce.job.combine.class
   * under the new API and from mapred.combiner.class otherwise (ConfigUtils.useNewApi).  A sum reducer over another
   * value class fails here instead of with a ClassCastException at the first spill.
   */
  static int combinerKind(Object combiner, Configuration conf) throws IOException {
    if (combiner == null || !combiner.getClass().getName().equals("org.apache.tez.mapreduce.combine.MRCombiner")) {
      return COMBINE_NONE;
    }
    final String reducer = conf.get(conf.getBoolean("mapred.mapper.new-api", false)
        ? "mapreduce.job.combine.class" : "mapred.combiner.class", "");
    final int kind;
    final String need;
    if (reducer.equals("org.apache.hadoop.mapreduce.lib.reduce.IntSumReducer")) {
      kind = COMBINE_INT_SUM;
      need = IntWritable.class.getName();
    } else if (reducer.equals("org.apache.hadoop.mapreduce.lib.reduce.LongSumReducer")
        || reducer.equals("org.apache.hadoop.mapred.lib.LongSumReducer")) {
      kind = COMBINE_LONG_SUM;
      need = LongWritable.class.getName();
    } else {
      return COMBINE_NONE;
    }
    final String val = ConfigUtils.getIntermediateOutputValueClass(conf).getName();
    if (!val.equals(need)) {
      throw new IOException("combiner " + reducer + " sums " + need + " values, but the value class is '" + val + "'");
    }
    return kind;
  }

  /** The device path supports a closed set of RawComparators; anything else keeps tez.runtime.sorter.class=PIPELINED. */
  static int comparatorId(RawComparator<?> c, Configuration conf) throws IOException {
    if (c instanceof TezBytesComparator) return CMP_BYTES;
    if (c instanceof Text.Comparator) return CMP_TEXT;
    if (c instanceof BytesWritable.Comparator) return CMP_BYTESWRITABLE;
    if (c instanceof IntWritable.Comparator) return CMP_INT;
    if (c instanceof LongWritable.Comparator) return CMP_LONG;
    throw new IOException("GpuSorter: no device comparator for " + c.getClass().getName()
        + " (supported: TezBytesComparator, Text, BytesWritable, IntWritable, LongWritable)");
  }

  @Override
  public void write(Object key, Object value) throws IOException {
    final int p = deviceHash ? -1 : partitioner.getPartition(key, value, partitions);
    if (!deviceHash && (p < 0 || p >= partitions)) {
      throw new IOException("Illegal partition for " + key + " (" + p + ")"); // PipelinedSorter.java:410-413
    }
    final int ks = kv.position();
    keySerializer.serialize(key); // the same serializers PipelinedSorter.collect drives
    final int vs = kv.position();
    valSerializer.serialize(value);
    keyOff.put(n, ks);
    valOff.put(n, vs);
    valLen.put(n, kv.position() - vs);
    if (!deviceHash) part.put(n, p);
    mapOutputRecordCounter.increment(1);
    mapOutputByteCounter.increment(kv.position() - ks);
    if (++n == BATCH_RECORDS || kv.remaining() < (BATCH_BYTES >> 3)) pushBatch();
    // the granted sort memory bounds what one spill holds (ExternalSorter.getInitialMemoryRequirement, :330-347)
    if (collectedBytes + kv.position() > availableMemoryMb * 1024L * 1024L) {
      pushBatch();
      spill(false);
    }
  }

  private void pushBatch() throws IOException {
    if (n == 0) return;
    nativeCollect(handle, kv, kv.position(), keyOff, valOff, valLen, deviceHash ? null : part, n); // tezgpu_sorter_collect_batch
    collectedBytes += kv.position();
    kv.clear();
    n = 0;
  }

  private void spill(boolean last) throws IOException {
    final org.apache.hadoop.fs.Path out = mapOutputFile.getSpillFileForWrite(numSpills, collectedBytes);
    final org.apache.hadoop.fs.Path index = mapOutputFile.getSpillIndexFileForWrite(numSpills, partitions * 24L + 8);
    final long[] idx = new long[3 * partitions];
    final long[] counters = new long[8];
    nativeFlush(handle, out.toString(), index.toString(), idx, counters); // tezgpu_sorter_flush: file.out + file.out.index, 0640
    nativeReset(handle);
    lastSpillRle = counters[5] != 0;                 // decided on the records before the combine
    outputBytesWithOverheadCounter.increment(counters[0]);
    spilledRecordsCounter.increment(counters[2]);   // after the combine: what the writer wrote
    if (combineKind != COMBINE_NONE) {
      final long[] info = new long[2];
      nativeCombineInfo(handle, info);              // tezgpu_sorter_combine_info
      // counted by MRCombiner's ValuesIterator and writer in the reference
      outputContext.getCounters().findCounter(TaskCounter.COMBINE_INPUT_RECORDS).increment(info[0]);
      outputContext.getCounters().findCounter(TaskCounter.COMBINE_OUTPUT_RECORDS).increment(info[1]);
    }
    if (reportPartitionStats()) {
      for (int i = 0; i < partitions; i++) partitionStats[i] += idx[3 * i + 1]; // PipelinedSorter.java:631-633
    }
    numSpills++;
    collectedBytes = 0;
  }

  @Override
  public void flush() throws IOException {
    pushBatch();
    spill(true);
    numAdditionalSpills.increment(numSpills - 1);
    if (numSpills == 1 || !isFinalMergeEnabled()) {
      // single spill: sameVolRename to the final names (PipelinedSorter.java:730-756) -- unchanged reference code
      finishSingleSpillOrPipelined();
      return;
    }
    // final merge of all spills on the device, every partition at once (PipelinedSorter.java:774-836):
    // checkForSameKeys and the writer's rle are both needsRLE() of the LAST spill (:797-814)
    finalOutputFile = mapOutputFile.getOutputFileForWrite(0);
    finalIndexFile = mapOutputFile.getOutputIndexFileForWrite(0);
    GpuMergeIterator.mergeSpillsToFile(spillFilePaths(), spillIndexPaths(), partitions,
        comparatorId(comparator, conf), sendEmptyPartitionDetails, lastSpillRle, lastSpillRle,
        numSpills >= minSpillsForCombine ? combineKind : COMBINE_NONE, finalOutputFile.toString(),
        finalIndexFile.toString());
    numShuffleChunks.setValue(1);
  }

  @Override
  public void close() throws IOException {
    super.close();
    if (handle != 0) nativeDestroy(handle);
    handle = 0;
  }

  // helpers a maintainer wires to the reference's own code (names as in PipelinedSorter)
  private void finishSingleSpillOrPipelined() throws IOException { /* PipelinedSorter.flush :730-772 */ }
  private String[] spillFilePaths() { return new String[numSpills]; }
  private String[] spillIndexPaths() { return new String[numSpills]; }

  // every native failure surfaces as IOException(tezgpu_last_error()), like the reference's own failures
  private static native long nativeCreate(int partitions, int comparator, int partitioner, boolean sendEmpty, long memory,
      int device) throws IOException;
  private static native void nativeCollect(long h, ByteBuffer kv, int bytes, IntBuffer keyOff, IntBuffer valOff,
      IntBuffer valLen, IntBuffer partition, int n) throws IOException;
  /** counters: [0] OUTPUT_BYTES_WITH_OVERHEAD [1] OUTPUT_BYTES_PHYSICAL [2] SPILLED_RECORDS [3] OUTPUT_RECORDS
   *  [4] OUTPUT_BYTES [5] rle used [6] adjacent equal keys [7] kernel launches */
  private static native void nativeFlush(long h, String out, String index, long[] idx, long[] counters) throws IOException;
  private static native void nativeReset(long h) throws IOException;
  private static native void nativeSetCombiner(long h, int kind) throws IOException;
  /** info: [0] records into, [1] records out of the last flush's combine */
  private static native void nativeCombineInfo(long h, long[] info) throws IOException;
  private static native void nativeDestroy(long h);

  /** DataOutputStream target that appends to the direct batch buffer. */
  private static final class ByteBufferOutputStream extends java.io.OutputStream {
    private final ByteBuffer b;
    ByteBufferOutputStream(ByteBuffer b) { this.b = b; }
    @Override public void write(int v) { b.put((byte) v); }
    @Override public void write(byte[] a, int off, int len) { b.put(a, off, len); }
  }
}
