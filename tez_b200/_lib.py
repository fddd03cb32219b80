"""ctypes loader for libtezgpu.so.  Fails loudly: there is no Python/CPU fallback for the hot path."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# TEZGPU_LIB: developer override to A/B another build of the same library (tools/variants/)
LIB_PATH = os.environ.get("TEZGPU_LIB") or os.path.join(HERE, "libtezgpu.so")


class Conf(C.Structure):
    """tezgpu_conf (include/tezgpu.h)"""
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("num_partitions", C.c_int32),
                ("comparator", C.c_int32), ("partitioner", C.c_int32), ("rle_policy", C.c_int32),
                ("send_empty_partition_details", C.c_int32), ("sorter_impl", C.c_int32),
                ("fixed_key_len", C.c_uint32), ("fixed_val_len", C.c_uint32), ("mem_budget_bytes", C.c_uint64)]


class WireSegment(C.Structure):
    """tezgpu_wire_segment (include/tezgpu.h)"""
    _fields_ = [("map_id", C.c_char * 1008), ("part_len", C.c_int64), ("raw_len", C.c_int64), ("offset", C.c_uint64),
                ("reduce", C.c_int32), ("reserved", C.c_int32)]


class Stats(C.Structure):
    """tezgpu_stats (include/tezgpu.h)"""
    _fields_ = [("output_records", C.c_int64), ("output_bytes", C.c_int64), ("output_bytes_with_overhead", C.c_int64),
                ("output_bytes_physical", C.c_int64), ("spilled_records", C.c_int64), ("file_out_bytes", C.c_int64),
                ("num_spills", C.c_int32), ("rle_used", C.c_int32), ("adjacent_equal_keys", C.c_int64),
                ("tie_records", C.c_int64), ("ms_stage", C.c_float), ("ms_sort", C.c_float), ("ms_ties", C.c_float),
                ("ms_emit", C.c_float), ("ms_total", C.c_float), ("kernel_launches", C.c_int32), ("ms_emit_kernel", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if not k.startswith("reserved")}


class Segment(C.Structure):
    _fields_ = [("data", C.c_void_p), ("len", C.c_uint64), ("flags", C.c_uint32), ("partition", C.c_uint32)]


class CopyRange(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("len", C.c_uint64)]


class KvIndex(C.Structure):
    _fields_ = [("key_off", C.c_uint32), ("key_len", C.c_uint32), ("val_off", C.c_uint32), ("val_len", C.c_uint32),
                ("same_key", C.c_uint32)]


# every symbol include/tezgpu.h declares: (name, restype, argtypes)
_V, _P = C.c_void_p, C.POINTER
SYMBOLS = [
    ("tezgpu_last_error", C.c_char_p, []),
    ("tezgpu_abi_version", C.c_int32, []),
    ("tezgpu_device_count", C.c_int32, []),
    ("tezgpu_sorter_create", C.c_int32, [_P(Conf), _P(_V)]),
    ("tezgpu_sorter_collect_batch", C.c_int32, [_V, _V, C.c_uint64, _V, _V, _V, _V, C.c_uint32]),
    ("tezgpu_sorter_collect_fixed", C.c_int32, [_V, _V, _V, C.c_uint64]),
    ("tezgpu_sorter_flush", C.c_int32, [_V, C.c_char_p, C.c_char_p, _V, _P(Stats)]),
    ("tezgpu_sorter_flush_to_memory", C.c_int32, [_V, _V, C.c_uint64, _P(C.c_uint64), _V, _V, _P(Stats)]),
    ("tezgpu_sorter_output_bound", C.c_uint64, [_V]),
    ("tezgpu_sorter_destroy", C.c_int32, [_V]),
    ("tezgpu_sorter_reset", C.c_int32, [_V]),
    ("tezgpu_sorter_sort_device_fixed", C.c_int32, [_V, _V, _V, C.c_uint64, _V, C.c_uint64, _P(C.c_uint64), _V, _P(Stats)]),
    ("tezgpu_sorter_stream", _V, [_V]),
    ("tezgpu_sorter_set_combiner", C.c_int32, [_V, C.c_int32]),
    ("tezgpu_sorter_combine_info", C.c_int32, [_V, _P(C.c_uint64), _P(C.c_uint64), _P(C.c_float)]),
    ("tezgpu_shuffle_header_size", C.c_uint64, [C.c_char_p, C.c_int64, C.c_int64, C.c_int32]),
    ("tezgpu_shuffle_header_write", C.c_int32, [C.c_char_p, C.c_int64, C.c_int64, C.c_int32, _V, C.c_uint64, _P(C.c_uint64)]),
    ("tezgpu_shuffle_header_read", C.c_int32, [_V, C.c_uint64, _V, C.c_uint64, _P(C.c_int64), _P(C.c_int64), _P(C.c_int32), _P(C.c_uint64)]),
    ("tezgpu_shuffle_serve_bound", C.c_uint64, [C.c_char_p, _V, C.c_int32, C.c_int32]),
    ("tezgpu_shuffle_serve", C.c_int32, [C.c_int32, _V, _V, C.c_char_p, C.c_int32, C.c_int32, _V, C.c_uint64, _P(C.c_uint64), _V]),
    ("tezgpu_shuffle_receive", C.c_int32, [_V, C.c_uint64, _V, C.c_uint32, _P(C.c_uint32)]),
    ("tezgpu_debug_crc_emulate", C.c_uint32, [_V, C.c_uint64, C.c_uint32, C.c_uint32]),
    ("tezgpu_debug_chunk_fold_emulate", C.c_uint32, [_V, C.c_uint32, C.c_int32]),
    ("tezgpu_debug_runs_assemble_emulate", C.c_uint32, [_V, C.c_uint32, _V, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, _V, C.c_uint32]),
    ("tezgpu_debug_assemble_emulate", C.c_uint32, [_V, C.c_uint32, C.c_uint32, _V, C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, _V, C.c_uint32]),
    ("tezgpu_merge_open", C.c_int32, [_P(Conf), _P(Segment), C.c_uint32, _P(_V)]),
    ("tezgpu_merge_reopen", C.c_int32, [_V, _P(Segment), C.c_uint32]),
    ("tezgpu_merge_set_check_for_same_keys", C.c_int32, [_V, C.c_int32]),
    ("tezgpu_merge_parse_info", C.c_int32, [_V, _V, _V]),
    ("tezgpu_merge_counts", C.c_int32, [_V, _P(C.c_uint64), _P(C.c_uint64)]),
    ("tezgpu_merge_next_batch", C.c_int32, [_V, _V, C.c_uint64, _P(KvIndex), C.c_uint32, _P(C.c_uint32)]),
    ("tezgpu_merge_write_ifile", C.c_int32, [_V, C.c_char_p, _V, C.c_uint64, C.c_int32, _P(C.c_int64), _P(C.c_int64), _P(Stats)]),
    ("tezgpu_merge_output_bound", C.c_uint64, [_V]),
    ("tezgpu_merge_write_ifile_device", C.c_int32, [_V, _V, C.c_uint64, C.c_int32, _P(C.c_int64), _P(C.c_int64), _P(Stats)]),
    ("tezgpu_merge_write_partitions_device", C.c_int32, [_V, _V, C.c_uint64, C.c_int32, _P(C.c_uint64), _V, _P(Stats)]),
    ("tezgpu_merge_write_partitions", C.c_int32, [_V, C.c_char_p, C.c_char_p, C.c_int32, _V, _P(Stats)]),
    ("tezgpu_merge_set_combiner", C.c_int32, [_V, C.c_int32]),
    ("tezgpu_merge_combine_info", C.c_int32, [_V, _P(C.c_uint64), _P(C.c_uint64), _P(C.c_float)]),
    ("tezgpu_merge_stream", _V, [_V]),
    ("tezgpu_peer_alloc", C.c_int32, [C.c_int32, C.c_uint64, _P(_V), _V]),
    ("tezgpu_peer_free", C.c_int32, [C.c_int32, _V]),
    ("tezgpu_peer_open", C.c_int32, [C.c_int32, _V, _P(_V)]),
    ("tezgpu_peer_close", C.c_int32, [C.c_int32, _V]),
    ("tezgpu_fetch_ranges", C.c_int32, [C.c_int32, _P(CopyRange), C.c_uint32, _V, _P(C.c_float)]),
    ("tezgpu_fetch_segments_verified", C.c_int32, [C.c_int32, _V, C.c_uint32, _V, _P(C.c_float)]),
    ("tezgpu_merge_close", C.c_int32, [_V]),
]

RT_SYMBOLS = [
    ("tezrt_last_error", C.c_char_p, []),
    ("tezrt_output_create", C.c_int32, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, _P(_V)]),
    ("tezrt_output_initialize", C.c_int32, [_V, _P(C.c_int64)]),
    ("tezrt_output_memory_assigned", C.c_int32, [_V, C.c_int64]),
    ("tezrt_output_start", C.c_int32, [_V]),
    ("tezrt_output_write", C.c_int32, [_V, C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32, C.c_int32]),
    ("tezrt_output_close", C.c_int32, [_V, _P(C.c_int32)]),
    ("tezrt_output_event", C.c_int32, [_V, C.c_int32, _P(C.c_int32), _P(_V), _P(C.c_uint64), _P(C.c_int32), _P(C.c_int32)]),
    ("tezrt_output_counter", C.c_int64, [_V, C.c_char_p]),
    ("tezrt_output_num_spills", C.c_int32, [_V]),
    ("tezrt_output_file", C.c_char_p, [_V]),
    ("tezrt_output_index_file", C.c_char_p, [_V]),
    ("tezrt_output_destroy", C.c_int32, [_V]),
    ("tezrt_input_create", C.c_int32, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_int64, C.c_int32, C.c_int32, _P(_V)]),
    ("tezrt_input_initialize", C.c_int32, [_V, _P(C.c_int64)]),
    ("tezrt_input_start", C.c_int32, [_V]),
    ("tezrt_input_add_local_output", C.c_int32, [_V, C.c_int32, C.c_char_p, C.c_char_p, C.c_int32, C.c_int32]),
    ("tezrt_input_add_local_spill", C.c_int32, [_V, C.c_int32, C.c_char_p, C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    ("tezrt_input_wait_ready", C.c_int32, [_V]),
    ("tezrt_input_next", C.c_int32, [_V, _P(_V), _P(C.c_uint32)]),
    ("tezrt_input_next_value", C.c_int32, [_V, _P(_V), _P(C.c_uint32)]),
    ("tezrt_input_counter", C.c_int64, [_V, C.c_char_p]),
    ("tezrt_input_destroy", C.c_int32, [_V]),
]

_lib = None


def load():
    """Returns the loaded library; raises if the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "tez_b200: %s is missing -- build it with `python -m tez_b200.build` "
                "(the hot path has no Python or CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS + RT_SYMBOLS:
            fn = getattr(L, name)  # AttributeError if the ABI and the header drift apart
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class TezGpuError(IOError):
    """Every failure of the path surfaces as an IOException in the reference (SURVEY 8b); same here."""

    def __init__(self, code, msg):
        super().__init__("tezgpu error %d: %s" % (code, msg))
        self.code = code


def check(rc):
    if rc != 0:
        raise TezGpuError(rc, load().tezgpu_last_error().decode("utf-8", "replace"))


def check_rt(rc):
    if rc != 0:
        raise TezGpuError(rc, load().tezrt_last_error().decode("utf-8", "replace"))
