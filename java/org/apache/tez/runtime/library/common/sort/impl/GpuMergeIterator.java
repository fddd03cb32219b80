/*
 * GpuMergeIterator -- TezMerger.merge(...) -> TezRawKeyValueIterator on the device (include/tezgpu.h, tezgpu_merge_*).
 *
 * Replaces the MergeQueue the reference builds at OG/MergeManager.java:804-811,899-903,1035-1041,1197-1199,1301-1319
 * and in PipelinedSorter.flush (:797-806).  NOT COMPILED IN THIS REPOSITORY (no JDK in the build image); the native side
 * is jni/tezgpu_jni.c.
 */
package org.apache.tez.runtime.library.common.sort.impl;

import java.io.IOException;
import java.nio.ByteBuffer;
import java.nio.ByteOrder;
import java.nio.IntBuffer;

import org.apache.hadoop.io.DataInputBuffer;
import org.apache.hadoop.util.Progress;

public final class GpuMergeIterator implements TezRawKeyValueIterator {
  static {
    System.loadLibrary("tezgpu_jni");
  }

  static final int SEG_HAS_HEADER = 1, SEG_DEVICE = 2, SEG_VERIFIED = 4;
  private static final int BATCH_BYTES = 8 << 20, BATCH_RECORDS = 1 << 16;

  private long handle; // tezgpu_merger*
  private final ByteBuffer batch = ByteBuffer.allocateDirect(BATCH_BYTES).order(ByteOrder.nativeOrder());
  private final IntBuffer idx = ByteBuffer.allocateDirect(5 * 4 * BATCH_RECORDS).order(ByteOrder.nativeOrder()).asIntBuffer();
  private final byte[] heap = new byte[BATCH_BYTES];   // DataInputBuffer wants a byte[]
  private final DataInputBuffer key = new DataInputBuffer(), value = new DataInputBuffer();
  private final Progress progress = new Progress();
  private int n, i = -1;

  /**
   * @param addresses  native addresses of the segments (in-memory byte[] pinned by the caller, or mapped file ranges)
   * @param lengths    segment lengths: header + body + 4 checksum bytes (partLength of the TezIndexRecord)
   * @param flags      SEG_HAS_HEADER for DiskSegments, 0 for InMemoryReader segments, | SEG_VERIFIED when the fetcher
   *                   already checked the CRC (IFile.Reader.readToMemory, IFile.java:764-809)
   * @param checkForSameKeys MergeQueue's constructor argument (TezMerger.java:560-573)
   */
  public GpuMergeIterator(long[] addresses, long[] lengths, int[] flags, int comparator, boolean checkForSameKeys)
      throws IOException {
    handle = nativeOpen(addresses, lengths, flags, null, 1, comparator, Integer.parseInt(System.getenv().getOrDefault("TEZGPU_DEVICE", "0")));
    if (!checkForSameKeys) nativeSetCheckForSameKeys(handle, false);
  }

  @Override
  public boolean next() throws IOException {
    if (++i >= n) {
      n = nativeNextBatch(handle, batch, BATCH_BYTES, idx, BATCH_RECORDS); // tezgpu_merge_next_batch
      i = 0;
      if (n > 0) {
        batch.position(0);
        batch.get(heap, 0, idx.get(5 * (n - 1) + 2) + idx.get(5 * (n - 1) + 3));
      }
    }
    return n > 0;
  }

  @Override public DataInputBuffer getKey() { key.reset(heap, idx.get(5 * i), idx.get(5 * i + 1)); return key; }
  @Override public DataInputBuffer getValue() { value.reset(heap, idx.get(5 * i + 2), idx.get(5 * i + 3)); return value; }
  @Override public boolean isSameKey() { return idx.get(5 * i + 4) != 0; }
  @Override public boolean hasNext() throws IOException { return i + 1 < n || nativeHasMore(handle); }
  @Override public Progress getProgress() { return progress; }

  /** TezMerger.writeFile(this, new IFile.Writer(..., rle)) collapses to one native call (TezMerger.java:215-245). */
  public long[] writeFile(String path, boolean writerRle) throws IOException {
    final long[] rawAndPart = new long[2];
    nativeWriteIFile(handle, path, writerRle, rawAndPart); // tezgpu_merge_write_ifile
    return rawAndPart;
  }

  @Override
  public void close() throws IOException {
    if (handle != 0) nativeClose(handle);
    handle = 0;
  }

  /** PipelinedSorter.flush's final merge: all spills, all partitions, one device pass (PipelinedSorter.java:774-836). */
  static void mergeSpillsToFile(String[] spillFiles, String[] spillIndexFiles, int partitions, int comparator,
      boolean sendEmptyPartitionDetails, boolean checkForSameKeys, boolean writerRle, int combiner, String out,
      String index) throws IOException {
    // combiner: GpuSorter.COMBINE_*, NONE unless numSpills >= tez.runtime.combine.min.spills (PipelinedSorter.java:815-820)
    nativeMergeSpills(spillFiles, spillIndexFiles, partitions, comparator, sendEmptyPartitionDetails, checkForSameKeys,
        writerRle, combiner, out, index); // tezgpu_merge_open(P) + set_check_for_same_keys + set_combiner + write_partitions
  }

  /** Combiner of writeFile (a MergeManager mem->disk merge that runs the combiner, OG/MergeManager.java:899-911). */
  void setCombiner(int kind) throws IOException {
    nativeSetCombiner(handle, kind); // tezgpu_merge_set_combiner
  }

  private static native long nativeOpen(long[] addresses, long[] lengths, int[] flags, int[] partitions, int numPartitions,
      int comparator, int device) throws IOException;
  private static native void nativeSetCheckForSameKeys(long h, boolean on) throws IOException;
  private static native int nativeNextBatch(long h, ByteBuffer out, int cap, IntBuffer idx, int idxCap) throws IOException;
  private static native boolean nativeHasMore(long h);
  private static native void nativeWriteIFile(long h, String path, boolean rle, long[] rawAndPart) throws IOException;
  private static native void nativeMergeSpills(String[] files, String[] indexFiles, int partitions, int comparator,
      boolean sendEmpty, boolean checkForSameKeys, boolean writerRle, int combiner, String out, String index)
      throws IOException;
  private static native void nativeSetCombiner(long h, int kind) throws IOException;
  private static native void nativeClose(long h);
}
