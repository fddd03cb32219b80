"""Thin object wrappers over the C ABI (include/tezgpu.h) -- what the JNI shim does in a Tez task JVM.

GpuSorter  ~ ExternalSorter seam (SORT/ExternalSorter.java:74-92): write/collect -> flush -> close.
GpuMerger  ~ TezMerger.merge(...) -> TezRawKeyValueIterator (SORT/TezMerger.java:717-912).
"""
import ctypes as C

import numpy as np

from . import _lib
from .constants import *  # noqa: F401,F403
from ._lib import Conf, KvIndex, Segment, Stats, check


def _ptr(a):
    return None if a is None else a.ctypes.data


def make_conf(num_partitions, comparator=CMP_BYTES, partitioner=PART_HASH, rle_policy=RLE_AUTO, send_empty=True,
              fixed=None, device=0, legacy=False, mem_budget=0, unordered=False):
    c = Conf()
    c.abi_version = ABI_VERSION
    c.device = device
    c.num_partitions = num_partitions
    c.comparator = comparator
    c.partitioner = partitioner
    c.rle_policy = rle_policy
    c.send_empty_partition_details = 1 if send_empty else 0
    c.sorter_impl = SORTER_UNORDERED if unordered else (SORTER_LEGACY if legacy else SORTER_PIPELINED)
    c.fixed_key_len, c.fixed_val_len = fixed if fixed else (0, 0)
    c.mem_budget_bytes = mem_budget
    return c


def _combine_info(fn, h):
    i, o, ms = C.c_uint64(), C.c_uint64(), C.c_float()
    check(fn(h, C.byref(i), C.byref(o), C.byref(ms)))
    return i.value, o.value, ms.value


class GpuSorter:
    def __init__(self, num_partitions, combiner=COMBINE_NONE, **kw):
        self.L = _lib.load()
        self.conf = make_conf(num_partitions, **kw)
        self.P = num_partitions
        self.h = C.c_void_p()
        check(self.L.tezgpu_sorter_create(C.byref(self.conf), C.byref(self.h)))
        if combiner != COMBINE_NONE:
            self.set_combiner(combiner)

    def set_combiner(self, kind):
        """COMBINE_INT_SUM / COMBINE_LONG_SUM: every flush writes one record per group of equal keys with the summed
        value (MRCombiner + IntSumReducer / LongSumReducer).  Before the first collect or right after reset()."""
        check(self.L.tezgpu_sorter_set_combiner(self.h, kind))

    def combine_info(self):
        """(records into, records out of, device ms of) the combine of the last flush."""
        return _combine_info(self.L.tezgpu_sorter_combine_info, self.h)

    def close(self):
        if self.h:
            self.L.tezgpu_sorter_destroy(self.h)
            self.h = C.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def collect(self, kv, key_off, val_off, val_len, partition=None):
        kv = np.ascontiguousarray(np.frombuffer(kv, dtype=np.uint8) if isinstance(kv, (bytes, bytearray)) else kv,
                                  dtype=np.uint8)
        key_off = np.ascontiguousarray(key_off, dtype=np.uint32)
        val_off = np.ascontiguousarray(val_off, dtype=np.uint32)
        val_len = np.ascontiguousarray(val_len, dtype=np.uint32)
        if partition is not None:
            partition = np.ascontiguousarray(partition, dtype=np.int32)
        check(self.L.tezgpu_sorter_collect_batch(self.h, _ptr(kv), kv.size, _ptr(key_off), _ptr(val_off),
                                                 _ptr(val_len), _ptr(partition), len(key_off)))

    def collect_fixed(self, kv, partition=None, n=None):
        if isinstance(kv, int):  # raw host pointer (pinned memory)
            p = kv
        else:
            kv = np.ascontiguousarray(kv, dtype=np.uint8)
            p = kv.ctypes.data
            if n is None:
                n = kv.size // (self.conf.fixed_key_len + self.conf.fixed_val_len)
        if partition is not None:
            partition = np.ascontiguousarray(partition, dtype=np.int32)
        check(self.L.tezgpu_sorter_collect_fixed(self.h, p, _ptr(partition), n))

    def reset(self):
        check(self.L.tezgpu_sorter_reset(self.h))

    def output_bound(self):
        return self.L.tezgpu_sorter_output_bound(self.h)

    def flush_to_memory(self, out=None):
        """Returns (file_out uint8 array view, index_bytes, index[P,3], stats dict)."""
        if out is None:
            out = np.empty(self.output_bound(), dtype=np.uint8)
        cap = out.size
        n = C.c_uint64()
        index = np.zeros((self.P, 3), dtype=np.int64)
        index_bytes = np.zeros(self.P * 24 + 8, dtype=np.uint8)
        st = Stats()
        check(self.L.tezgpu_sorter_flush_to_memory(self.h, _ptr(out), cap, C.byref(n), _ptr(index_bytes), _ptr(index),
                                                   C.byref(st)))
        return out[:n.value], index_bytes.tobytes(), index, st.as_dict()

    def flush(self, out_path, index_path):
        index = np.zeros((self.P, 3), dtype=np.int64)
        st = Stats()
        check(self.L.tezgpu_sorter_flush(self.h, out_path.encode(), index_path.encode(), _ptr(index), C.byref(st)))
        return index, st.as_dict()

    def sort_device_fixed(self, d_kv, n, d_out, out_cap, d_partition=None):
        """Device-resident records (raw device pointers as ints). Returns (out_len, index, stats)."""
        out_len = C.c_uint64()
        index = np.zeros((self.P, 3), dtype=np.int64)
        st = Stats()
        check(self.L.tezgpu_sorter_sort_device_fixed(self.h, d_kv, d_partition, n, d_out, out_cap, C.byref(out_len),
                                                     _ptr(index), C.byref(st)))
        return out_len.value, index, st.as_dict()

    def stream(self):
        return self.L.tezgpu_sorter_stream(self.h)


class GpuMerger:
    def __init__(self, segments, comparator=CMP_BYTES, device=0, has_header=True, device_ptrs=False, fixed=None,
                 partitions=None, num_partitions=1, send_empty=True, verified=None):
        """segments: list of bytes / uint8 arrays (host) or (ptr, len) tuples when device_ptrs.
        verified: optional per-segment booleans -- the transport already checked that segment's checksum
        (TEZGPU_SEG_VERIFIED: fetch_segments_verified), the merge does not read it again to verify."""
        self.L = _lib.load()
        self.conf = make_conf(num_partitions, comparator=comparator, partitioner=PART_GIVEN, device=device, fixed=fixed,
                              send_empty=send_empty)
        self.P = num_partitions
        self._has_header, self._device_ptrs = has_header, device_ptrs
        arr = self._segments(segments, partitions, verified)
        self.h = C.c_void_p()
        check(self.L.tezgpu_merge_open(C.byref(self.conf), arr, len(segments), C.byref(self.h)))

    def _segments(self, segments, partitions, verified=None):
        self._keep = []
        arr = (Segment * max(1, len(segments)))()
        flags = (SEG_HAS_HEADER if self._has_header else 0) | (SEG_DEVICE if self._device_ptrs else 0)
        if self._device_ptrs and len(segments) > 64:
            # many device-resident runs (the reduce side of the multi-GPU shuffle): fill the table through numpy
            tab = np.zeros(len(segments), dtype=np.dtype([("data", "<u8"), ("len", "<u8"), ("flags", "<u4"), ("partition", "<u4")]))
            sp = np.asarray(segments, dtype=np.uint64).reshape(-1, 2)
            tab["data"], tab["len"], tab["flags"] = sp[:, 0], sp[:, 1], flags
            if verified is not None:
                tab["flags"] |= np.where(np.asarray(verified, dtype=bool), SEG_VERIFIED, 0).astype(np.uint32)
            if partitions is not None:
                tab["partition"] = np.asarray(partitions, dtype=np.uint32)
            self._keep.append(tab)
            return C.cast(tab.ctypes.data, C.POINTER(Segment))
        for i, s in enumerate(segments):
            if self._device_ptrs:
                arr[i].data, arr[i].len = s
            else:
                a = np.ascontiguousarray(np.frombuffer(s, dtype=np.uint8) if isinstance(s, (bytes, bytearray)) else s)
                self._keep.append(a)
                arr[i].data = a.ctypes.data if a.size else None
                arr[i].len = a.size
            arr[i].flags = flags | (SEG_VERIFIED if (verified is not None and verified[i]) else 0)
            arr[i].partition = 0 if partitions is None else int(partitions[i])
        return arr

    def reopen(self, segments, partitions=None, verified=None):
        """New merge through the same handle (device allocations are kept)."""
        arr = self._segments(segments, partitions, verified)
        check(self.L.tezgpu_merge_reopen(self.h, arr, len(segments)))

    def close(self):
        if self.h:
            self.L.tezgpu_merge_close(self.h)
            self.h = C.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_check_for_same_keys(self, on):
        """MergeQueue's checkForSameKeys (SORT/TezMerger.java:560-573); default True."""
        check(self.L.tezgpu_merge_set_check_for_same_keys(self.h, 1 if on else 0))

    def set_combiner(self, kind):
        """Combiner of the write_* calls (a combining final merge); records() stays the uncombined stream."""
        check(self.L.tezgpu_merge_set_combiner(self.h, kind))

    def combine_info(self):
        """(records into, records out of, device ms of) the combine of the last write."""
        return _combine_info(self.L.tezgpu_merge_combine_info, self.h)

    def parse_info(self):
        """(mode, windows walked by hand) of the last open: 0 records addressed in place, 1 window parser, 2 sequential walker."""
        m, r = C.c_int32(), C.c_int32()
        check(self.L.tezgpu_merge_parse_info(self.h, C.byref(m), C.byref(r)))
        return m.value, r.value

    def counts(self):
        r, b = C.c_uint64(), C.c_uint64()
        check(self.L.tezgpu_merge_counts(self.h, C.byref(r), C.byref(b)))
        return r.value, b.value

    def records(self, batch_records=1 << 16, batch_bytes=1 << 24):
        """Iterates (key, value, is_same_key) like TezRawKeyValueIterator.next/getKey/getValue/isSameKey."""
        buf = np.empty(batch_bytes, dtype=np.uint8)
        idx = (KvIndex * batch_records)()
        n = C.c_uint32()
        while True:
            check(self.L.tezgpu_merge_next_batch(self.h, _ptr(buf), buf.size, idx, batch_records, C.byref(n)))
            if n.value == 0:
                return
            raw = buf.tobytes()
            for i in range(n.value):
                e = idx[i]
                yield (raw[e.key_off:e.key_off + e.key_len], raw[e.val_off:e.val_off + e.val_len], bool(e.same_key))

    def output_bound(self):
        return self.L.tezgpu_merge_output_bound(self.h)

    def write_ifile(self, rle=False, path=None):
        """TezMerger.writeFile into an IFile.Writer(rle). Returns (segment bytes or None, rawLen, partLen, stats)."""
        raw, part = C.c_int64(), C.c_int64()
        st = Stats()
        if path is not None:
            check(self.L.tezgpu_merge_write_ifile(self.h, path.encode(), None, 0, 1 if rle else 0, C.byref(raw),
                                                  C.byref(part), C.byref(st)))
            return None, raw.value, part.value, st.as_dict()
        out = np.empty(self.output_bound(), dtype=np.uint8)
        check(self.L.tezgpu_merge_write_ifile(self.h, None, _ptr(out), out.size, 1 if rle else 0, C.byref(raw),
                                              C.byref(part), C.byref(st)))
        return out[:part.value].tobytes(), raw.value, part.value, st.as_dict()

    def write_ifile_device(self, d_out, out_cap, rle=False):
        raw, part = C.c_int64(), C.c_int64()
        st = Stats()
        check(self.L.tezgpu_merge_write_ifile_device(self.h, d_out, out_cap, 1 if rle else 0, C.byref(raw),
                                                     C.byref(part), C.byref(st)))
        return raw.value, part.value, st.as_dict()

    def write_partitions_device(self, d_out, out_cap, rle=False):
        """Batched reduce side: P merged segments back to back. Returns (out_len, index[P,3], stats)."""
        n = C.c_uint64()
        index = np.zeros((self.P, 3), dtype=np.int64)
        st = Stats()
        check(self.L.tezgpu_merge_write_partitions_device(self.h, d_out, out_cap, 1 if rle else 0, C.byref(n), _ptr(index),
                                                          C.byref(st)))
        return n.value, index, st.as_dict()

    def stream(self):
        return self.L.tezgpu_merge_stream(self.h)


class PeerBuffer:
    """Device buffer other processes of the box can map (tezgpu_peer_alloc): where a producer keeps file.out."""

    def __init__(self, nbytes, device=0):
        self.L = _lib.load()
        self.device, self.nbytes = device, int(nbytes)
        p = C.c_void_p()
        handle = (C.c_uint8 * 64)()
        check(self.L.tezgpu_peer_alloc(device, self.nbytes, C.byref(p), handle))
        self.ptr, self.handle = p.value, bytes(handle)

    def close(self):
        if self.ptr:
            check(self.L.tezgpu_peer_free(self.device, self.ptr))
            self.ptr = None


class PeerMapping:
    """A peer's exported buffer mapped into this process (tezgpu_peer_open)."""

    def __init__(self, handle, device=0):
        self.L = _lib.load()
        self.device = device
        p = C.c_void_p()
        buf = (C.c_uint8 * 64).from_buffer_copy(handle)
        check(self.L.tezgpu_peer_open(device, buf, C.byref(p)))
        self.ptr = p.value

    def close(self):
        if self.ptr:
            check(self.L.tezgpu_peer_close(self.device, self.ptr))
            self.ptr = None


FETCH_SEG_DTYPE = np.dtype([("src", "<u8"), ("dst", "<u8"), ("len", "<u8"), ("flags", "<u4"), ("reserved", "<u4")])


def fetch_segments_verified(segs, device=0, stream=None, has_header=True):
    """segs: iterable of (src_ptr, dst_ptr, nbytes) -- one IFile segment each.  One launch copies them and verifies every
    segment's CRC32 trailer on the bytes in flight (IFile.Reader.readToMemory); raises TezGpuError(TEZGPU_E_FORMAT) on a
    mismatch.  Returns the copy kernel's time in ms."""
    L = _lib.load()
    tab = np.zeros(len(segs), dtype=FETCH_SEG_DTYPE)
    if len(segs):
        a = np.asarray(segs, dtype=np.uint64).reshape(-1, 3)
        tab["src"], tab["dst"], tab["len"] = a[:, 0], a[:, 1], a[:, 2]
        tab["flags"] = SEG_HAS_HEADER if has_header else 0
    ms = C.c_float()
    check(L.tezgpu_fetch_segments_verified(device, tab.ctypes.data, len(segs), stream, C.byref(ms)))
    return ms.value


def fetch_ranges(ranges, device=0, stream=None):
    """ranges: list of (src_ptr, dst_ptr, nbytes) device addresses; one launch, returns the kernel time in ms."""
    L = _lib.load()
    arr = (_lib.CopyRange * max(1, len(ranges)))()
    for i, (s, d, n) in enumerate(ranges):
        arr[i].src, arr[i].dst, arr[i].len = s, d, n
    ms = C.c_float()
    check(L.tezgpu_fetch_ranges(device, arr, len(ranges), stream, C.byref(ms)))
    return ms.value


# ---------------------------------------------------------------- SURVEY 8 f-2: ShuffleHandler <-> fetcher wire format
def shuffle_header(map_id, part_len, raw_len, reduce):
    """ShuffleHeader.write (OG/ShuffleHeader.java:101-106) -> bytes."""
    L = _lib.load()
    mid = map_id.encode("utf-8")
    buf = (C.c_uint8 * (len(mid) + 64))()
    n = C.c_uint64()
    check(L.tezgpu_shuffle_header_write(mid, part_len, raw_len, reduce, buf, len(buf), C.byref(n)))
    assert n.value == L.tezgpu_shuffle_header_size(mid, part_len, raw_len, reduce)
    return bytes(buf[:n.value])


def read_shuffle_header(data):
    """ShuffleHeader.readFields -> (map_id, part_len, raw_len, reduce, header bytes consumed)."""
    L = _lib.load()
    mid = C.create_string_buffer(1008)
    pl, rl, rd, used = C.c_int64(), C.c_int64(), C.c_int32(), C.c_uint64()
    raw = bytes(data)
    check(L.tezgpu_shuffle_header_read(raw, len(raw), mid, len(mid), C.byref(pl), C.byref(rl), C.byref(rd), C.byref(used)))
    return mid.value.decode("utf-8"), pl.value, rl.value, rd.value, used.value


def shuffle_serve(d_file_out, index, map_id, reduce0, nreduce, device=0, stream=None):
    """Response body ShuffleHandler sends for reducers [reduce0, reduce0 + nreduce) of one map output whose file.out is in
    device memory (d_file_out = device pointer, index = (P, 3) int64 spill index) -> bytes."""
    L = _lib.load()
    idx = np.ascontiguousarray(index, dtype=np.int64)
    mid = map_id.encode("utf-8")
    cap = L.tezgpu_shuffle_serve_bound(mid, idx.ctypes.data, reduce0, nreduce)
    out = np.empty(max(1, cap), dtype=np.uint8)
    n = C.c_uint64()
    check(L.tezgpu_shuffle_serve(device, d_file_out, idx.ctypes.data, mid, reduce0, nreduce, out.ctypes.data, cap, C.byref(n), stream))
    return out[:n.value].tobytes()


def shuffle_receive(body):
    """Splits a response body into [(map_id, reduce, raw_len, segment bytes)] the way FetcherOrderedGrouped.copyMapOutput
    walks it (header, then compressedLength bytes)."""
    L = _lib.load()
    raw = bytes(body)
    n = C.c_uint32()
    cap = 64
    while True:
        tab = (_lib.WireSegment * cap)()
        rc = L.tezgpu_shuffle_receive(raw, len(raw), tab, cap, C.byref(n))
        if rc != 0 and n.value > cap:
            cap = n.value
            continue
        check(rc)
        break
    return [(s.map_id.decode("utf-8"), s.reduce, s.raw_len, raw[s.offset:s.offset + s.part_len]) for s in tab[:n.value]]
