/*
 * tezgpu_jni.c -- JNI shim between the Java bindings (java/.../GpuSorter.java, GpuMergeIterator.java) and the C ABI of
 * libtezgpu.so (include/tezgpu.h).  Thin on purpose: direct ByteBuffers in, error codes out as java.io.IOException with
 * tezgpu_last_error() as the message (every failure of the reference path is an IOException too).
 *
 * build (where a JDK exists):
 *   gcc -shared -fPIC -I$JAVA_HOME/include -I$JAVA_HOME/include/linux -Iinclude jni/tezgpu_jni.c \
 *       -Ltez_b200 -ltezgpu -o libtezgpu_jni.so
 * The build image of this repository has no JDK: this file is syntax-checked against a minimal jni.h stand-in only.
 */
#include <jni.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "tezgpu.h"

#define SORTER(fn) Java_org_apache_tez_runtime_library_common_sort_impl_GpuSorter_##fn
#define MERGER(fn) Java_org_apache_tez_runtime_library_common_sort_impl_GpuMergeIterator_##fn

static void throw_io(JNIEnv *env, const char *msg) {
  jclass c = (*env)->FindClass(env, "java/io/IOException");
  if (c) (*env)->ThrowNew(env, c, msg ? msg : "tezgpu failure");
}
static int failed(JNIEnv *env, int32_t rc) {
  if (rc == TEZGPU_OK) return 0;
  throw_io(env, tezgpu_last_error());
  return 1;
}
static void *addr(JNIEnv *env, jobject buf) { return buf ? (*env)->GetDirectBufferAddress(env, buf) : NULL; }

/* ------------------------------------------------------------------------------------------------ GpuSorter */
JNIEXPORT jlong JNICALL SORTER(nativeCreate)(JNIEnv *env, jclass cls, jint partitions, jint comparator, jint partitioner,
                                             jboolean send_empty, jlong memory, jint device) {
  (void)cls;
  tezgpu_conf c;
  memset(&c, 0, sizeof(c));
  c.abi_version = TEZGPU_ABI_VERSION;
  c.device = device;
  c.num_partitions = partitions;
  c.comparator = comparator;
  c.partitioner = partitioner;
  c.rle_policy = TEZGPU_RLE_AUTO;
  c.send_empty_partition_details = send_empty ? 1 : 0;
  c.mem_budget_bytes = (uint64_t)memory;
  tezgpu_sorter *h = NULL;
  if (failed(env, tezgpu_sorter_create(&c, &h))) return 0;
  return (jlong)(intptr_t)h;
}

JNIEXPORT void JNICALL SORTER(nativeCollect)(JNIEnv *env, jclass cls, jlong h, jobject kv, jint bytes, jobject key_off,
                                             jobject val_off, jobject val_len, jobject partition, jint n) {
  (void)cls;
  failed(env, tezgpu_sorter_collect_batch((tezgpu_sorter *)(intptr_t)h, (const uint8_t *)addr(env, kv), (uint64_t)bytes,
                                          (const uint32_t *)addr(env, key_off), (const uint32_t *)addr(env, val_off),
                                          (const uint32_t *)addr(env, val_len), (const int32_t *)addr(env, partition),
                                          (uint32_t)n));
}

JNIEXPORT void JNICALL SORTER(nativeFlush)(JNIEnv *env, jclass cls, jlong h, jstring out, jstring index, jlongArray idx,
                                           jlongArray counters) {
  (void)cls;
  const char *o = (*env)->GetStringUTFChars(env, out, NULL), *x = (*env)->GetStringUTFChars(env, index, NULL);
  jsize n3 = (*env)->GetArrayLength(env, idx);
  int64_t *tri = (int64_t *)calloc((size_t)n3 + 1, sizeof(int64_t));
  tezgpu_stats st;
  memset(&st, 0, sizeof(st));
  int32_t rc = tezgpu_sorter_flush((tezgpu_sorter *)(intptr_t)h, o, x, tri, &st);
  (*env)->ReleaseStringUTFChars(env, out, o);
  (*env)->ReleaseStringUTFChars(env, index, x);
  if (!failed(env, rc)) {
    jlong c[8] = {st.output_bytes_with_overhead, st.output_bytes_physical, st.spilled_records, st.output_records,
                  st.output_bytes, st.rle_used, st.adjacent_equal_keys, st.kernel_launches};
    (*env)->SetLongArrayRegion(env, idx, 0, n3, (const jlong *)tri);
    (*env)->SetLongArrayRegion(env, counters, 0, 8, c);
  }
  free(tri);
}

JNIEXPORT void JNICALL SORTER(nativeReset)(JNIEnv *env, jclass cls, jlong h) {
  (void)cls;
  failed(env, tezgpu_sorter_reset((tezgpu_sorter *)(intptr_t)h));
}

JNIEXPORT void JNICALL SORTER(nativeSetCombiner)(JNIEnv *env, jclass cls, jlong h, jint kind) {
  (void)cls;
  failed(env, tezgpu_sorter_set_combiner((tezgpu_sorter *)(intptr_t)h, kind));
}

JNIEXPORT void JNICALL SORTER(nativeCombineInfo)(JNIEnv *env, jclass cls, jlong h, jlongArray info) {
  (void)cls;
  uint64_t in = 0, out = 0;
  if (!failed(env, tezgpu_sorter_combine_info((tezgpu_sorter *)(intptr_t)h, &in, &out, NULL))) {
    jlong v[2] = {(jlong)in, (jlong)out};
    (*env)->SetLongArrayRegion(env, info, 0, 2, v);
  }
}

JNIEXPORT void JNICALL SORTER(nativeDestroy)(JNIEnv *env, jclass cls, jlong h) {
  (void)env; (void)cls;
  tezgpu_sorter_destroy((tezgpu_sorter *)(intptr_t)h);
}

/* ------------------------------------------------------------------------------------------------ GpuMergeIterator */
JNIEXPORT jlong JNICALL MERGER(nativeOpen)(JNIEnv *env, jclass cls, jlongArray addresses, jlongArray lengths, jintArray flags,
                                           jintArray partitions, jint num_partitions, jint comparator, jint device) {
  (void)cls;
  jsize n = (*env)->GetArrayLength(env, addresses);
  jlong *a = (*env)->GetLongArrayElements(env, addresses, NULL), *l = (*env)->GetLongArrayElements(env, lengths, NULL);
  jint *f = (*env)->GetIntArrayElements(env, flags, NULL);
  jint *p = partitions ? (*env)->GetIntArrayElements(env, partitions, NULL) : NULL;
  tezgpu_segment *segs = (tezgpu_segment *)calloc((size_t)n + 1, sizeof(tezgpu_segment));
  for (jsize i = 0; i < n; i++) {
    segs[i].data = (const void *)(intptr_t)a[i];
    segs[i].len = (uint64_t)l[i];
    segs[i].flags = (uint32_t)f[i];
    segs[i].partition = p ? (uint32_t)p[i] : 0u;
  }
  tezgpu_conf c;
  memset(&c, 0, sizeof(c));
  c.abi_version = TEZGPU_ABI_VERSION;
  c.device = device;
  c.num_partitions = num_partitions;
  c.comparator = comparator;
  c.partitioner = TEZGPU_PART_GIVEN;
  c.send_empty_partition_details = 1;
  tezgpu_merger *m = NULL;
  int32_t rc = tezgpu_merge_open(&c, segs, (uint32_t)n, &m);
  free(segs);
  (*env)->ReleaseLongArrayElements(env, addresses, a, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, lengths, l, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, flags, f, JNI_ABORT);
  if (p) (*env)->ReleaseIntArrayElements(env, partitions, p, JNI_ABORT);
  if (failed(env, rc)) return 0;
  return (jlong)(intptr_t)m;
}

JNIEXPORT void JNICALL MERGER(nativeSetCheckForSameKeys)(JNIEnv *env, jclass cls, jlong h, jboolean on) {
  (void)cls;
  failed(env, tezgpu_merge_set_check_for_same_keys((tezgpu_merger *)(intptr_t)h, on ? 1 : 0));
}

JNIEXPORT void JNICALL MERGER(nativeSetCombiner)(JNIEnv *env, jclass cls, jlong h, jint kind) {
  (void)cls;
  failed(env, tezgpu_merge_set_combiner((tezgpu_merger *)(intptr_t)h, kind));
}

JNIEXPORT jint JNICALL MERGER(nativeNextBatch)(JNIEnv *env, jclass cls, jlong h, jobject out, jint cap, jobject idx, jint idx_cap) {
  (void)cls;
  uint32_t n = 0;
  if (failed(env, tezgpu_merge_next_batch((tezgpu_merger *)(intptr_t)h, (uint8_t *)addr(env, out), (uint64_t)cap,
                                          (tezgpu_kv_index *)addr(env, idx), (uint32_t)idx_cap, &n)))
    return 0;
  return (jint)n;
}

JNIEXPORT jboolean JNICALL MERGER(nativeHasMore)(JNIEnv *env, jclass cls, jlong h) {
  (void)env; (void)cls;
  uint64_t records = 0, kv = 0;
  /* the iterator keeps its own cursor; "more" = the stream is not empty (callers pair hasNext() with next()) */
  return tezgpu_merge_counts((tezgpu_merger *)(intptr_t)h, &records, &kv) == TEZGPU_OK && records > 0;
}

JNIEXPORT void JNICALL MERGER(nativeWriteIFile)(JNIEnv *env, jclass cls, jlong h, jstring path, jboolean rle, jlongArray raw_and_part) {
  (void)cls;
  const char *p = (*env)->GetStringUTFChars(env, path, NULL);
  int64_t raw = 0, part = 0;
  int32_t rc = tezgpu_merge_write_ifile((tezgpu_merger *)(intptr_t)h, p, NULL, 0, rle ? 1 : 0, &raw, &part, NULL);
  (*env)->ReleaseStringUTFChars(env, path, p);
  if (!failed(env, rc)) {
    jlong v[2] = {raw, part};
    (*env)->SetLongArrayRegion(env, raw_and_part, 0, 2, v);
  }
}

JNIEXPORT void JNICALL MERGER(nativeClose)(JNIEnv *env, jclass cls, jlong h) {
  (void)env; (void)cls;
  tezgpu_merge_close((tezgpu_merger *)(intptr_t)h);
}

/* nativeMergeSpills (PipelinedSorter.flush's final merge) reads the spill files and their TezSpillRecord indexes and
 * builds the partition-tagged segment table exactly as tez_b200/csrc/host/tez_runtime_library.cc::GpuSorter::flush does
 * (:281-330): tezgpu_merge_open(conf with num_partitions = P) -> tezgpu_merge_set_check_for_same_keys(needsRLE) ->
 * tezgpu_merge_set_combiner(kind, when numSpills >= combine.min.spills) -> tezgpu_merge_write_partitions(out, index,
 * rle = needsRLE).  It is that C++ code behind a JNI signature; kept there so
 * the logic exists once and is exercised by tests/test_runtime_library_gpu.py. */
