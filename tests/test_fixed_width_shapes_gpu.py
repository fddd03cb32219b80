"""Fixed-width records across record shapes, input alignments and emit kernels, byte for byte against the oracle.

SortPipeline::emit_phase (tez_b200/csrc/sorter.cuh) picks one of several emit kernels from the record shape, the input
alignment, the run-length decision and a few environment switches.  Every case here runs under torch.profiler and
checks which emit kernel was launched against `expected_emit_kernel`, a restatement of that dispatch, so a parity case
cannot pass while the kernel it was written for never runs.

  A  map side, records collected from the host (16-byte aligned staging): unique keys, and repeated keys with RLE on
  B  map side, device-resident input at offsets from the start of a tensor (16-byte multiples; others are refused)
  C  reduce side in run-table mode (records addressed in place): host segments with and without header, device
     segments at every start address mod 16, several partitions with more runs in one than the runs kernel plans
  D  declared shapes the bytes contradict: the merge must leave run-table mode and still equal the oracle
  F  every emit switch, in a subprocess (switches are read once per process) over a reduced shape list

Shapes cover framing headers vint(klen) vint(vlen) of 2 to 5 bytes, 1 to 1374 16-byte pieces per record (cpr), both
sides of emit4_fits (k_emit_fast4: cpr <= 8 and a tile's pieces fit five gather rounds), of emit4u_max_recs (cpr <= 31)
and of fast_emit_fits (one record plus lead, header and EOF fit the 22016-byte tile image)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import tez_oracle as O
import tez_b200 as T

pytestmark = pytest.mark.gpu

# ---------------------------------------------------------------------------------------------------------- switches
SWITCHES = {  # switch -> (value the sweep sets, emit kernel that must run at least once with it)
    "TEZGPU_EMIT_TMA": ("1", "k_emit_tma"),
    "TEZGPU_EMIT_RUNS": ("1", "k_emit_runs"),
    "TEZGPU_EMIT_V2": ("1", "k_emit_fast<5,true>"),
    "TEZGPU_EMIT_SUBS": ("3", "k_emit_fast4<5,3>"),
    "TEZGPU_EMIT_PIPE_UNALIGNED": ("0", "k_emit_fast<5,false>"),
    "TEZGPU_NO_FAST_EMIT": ("1", "k_emit<true>"),
    "TEZGPU_EMIT_ROUND_FILL": ("1", "k_emit_fast4<5,1>"),
}
DEFAULT_PATH = {"k_emit_fast4<5,1>", "k_emit_fast<5,true>", "k_emit_fast4u<5>", "k_emit_fast<5,false>", "k_emit<true>"}


def _atoi(s):
    m = re.match(r"\s*([+-]?\d+)", s or "")
    return int(m.group(1)) if m else 0


def _env_flags(env=os.environ):
    """The switches as the library reads them (getenv / atoi)."""
    g = env.get
    return dict(
        tma=g("TEZGPU_EMIT_TMA") is not None and _atoi(g("TEZGPU_EMIT_TMA")) != 0,
        runs=g("TEZGPU_EMIT_RUNS") is not None and _atoi(g("TEZGPU_EMIT_RUNS")) != 0,
        v2=g("TEZGPU_EMIT_V2") is not None,
        subs3=g("TEZGPU_EMIT_SUBS") is not None and _atoi(g("TEZGPU_EMIT_SUBS")) == 3,
        pipe_u=not (g("TEZGPU_EMIT_PIPE_UNALIGNED") is not None and _atoi(g("TEZGPU_EMIT_PIPE_UNALIGNED")) == 0),
        no_fast=g("TEZGPU_NO_FAST_EMIT") is not None,
        round_fill=_atoi(g("TEZGPU_EMIT_ROUND_FILL")) if g("TEZGPU_EMIT_ROUND_FILL") is not None else 0,
    )


FLAGS = _env_flags()
ACTIVE_SWITCHES = [k for k in SWITCHES if k in os.environ]

# ------------------------------------------------------------------------------------------------------------ shapes
SHAPES = [(8, 8), (16, 64), (16, 112), (16, 128), (16, 240), (128, 128), (16, 480), (16, 496), (16, 2032), (16, 4080),
          (16, 4096), (16, 21968), (16, 21984), (16, 32752), (16, 70000), (10, 7), (3, 5), (200, 57)]
# with a switch set (the sweep's child processes): the shapes that reach each kernel and the edges the switches move
SWEEP_SHAPES = [(8, 8), (16, 64), (16, 128), (16, 496), (16, 2032), (16, 32752), (10, 7)]
MATRIX = SWEEP_SHAPES if ACTIVE_SWITCHES else SHAPES

FE_IMG_BYTES = 22016
FE_THREADS = 256
MAX_BYTES = 48 << 20   # kv bytes of the largest case


def vint_size(v):
    """WritableUtils.getVIntSize"""
    if -112 <= v <= 127:
        return 1
    if v < 0:
        v ^= -1
    return (v.bit_length() + 7) // 8 + 1


def rec_size(klen, vlen):
    return vint_size(klen) + vint_size(vlen) + klen + vlen


def emit4u_max_recs(cpr):
    w = cpr + 1
    return 0 if w > 32 else 5 * (FE_THREADS // 32) * (32 // w)


def emit4_fits(recs, cpr):
    return cpr <= 8 and recs * cpr <= 5 * FE_THREADS


def fast_emit_fits(rs):
    return rs + 15 + 4 + 2 <= FE_IMG_BYTES


def recs_per_tile(klen, vlen, aligned, flags=FLAGS):
    """SortPipeline::set_fixed_layout (without the opt-in runs kernel's branch)."""
    rs = rec_size(klen, vlen)
    r = max(1, min(256, (FE_IMG_BYTES - 32) // rs))
    fill = flags["round_fill"] != 0
    stride = klen + vlen
    if flags["pipe_u"] and stride >= 16 and stride % 16 == 0 and not aligned and emit4u_max_recs(stride // 16) >= 32:
        r = min(r, emit4u_max_recs(stride // 16))
        fill = True
    if fill and r >= 32:
        cap, best, best_eff = r, r, 0.0
        for x in range(cap, cap - cap // 10 - 1, -1):
            chunks = (x * rs + 15 + 4 + 2 + 15) // 16
            eff = x / ((chunks + FE_THREADS - 1) // FE_THREADS)
            if eff > best_eff:
                best, best_eff = x, eff
        r = best
    return r


def expected_emit_kernel(klen, vlen, aligned, fixed_emit=True, flags=FLAGS):
    """SortPipeline::emit_phase's choice.  aligned: packed records at a 16-byte aligned address (map side); the
    reduce side's run table is never `aligned`.  None where an opt-in kernel's own fit test decides (TMA, runs)."""
    if not fixed_emit:
        return "k_emit<false>"           # records written as repeats: variable framing
    stride, rs = klen + vlen, rec_size(klen, vlen)
    if not (stride >= 16 and stride % 16 == 0 and fast_emit_fits(rs)) or flags["no_fast"]:
        return "k_emit<true>"
    cpr, r = stride // 16, recs_per_tile(klen, vlen, aligned, flags)
    if aligned:
        if flags["tma"]:
            return None
        if emit4_fits(r, cpr) and not flags["v2"]:
            return "k_emit_fast4<5,3>" if flags["subs3"] else "k_emit_fast4<5,1>"
        return "k_emit_fast<5,true>"
    if flags["runs"]:
        return None
    if flags["pipe_u"] and r <= emit4u_max_recs(cpr):
        return "k_emit_fast4u<5>"
    return "k_emit_fast<5,false>"


# ----------------------------------------------------------------------------------------------------- kernel capture
_EMIT_RE = re.compile(r"k_emit(?:_fast4u|_fast4|_fast|_tma|_runs)?(?:<[^<>()]*>)?(?=\(|$)")
OBSERVED = {}      # case id -> emit kernels launched
EXPECTED = {}      # case id -> emit kernel expected_emit_kernel named (or None)
PROFILER_SAW_KERNELS = []


def emit_kernels(names):
    out = set()
    for nm in names:
        for m in _EMIT_RE.finditer(nm):
            out.add(m.group(0).replace(" ", ""))
    return out


class _Launches:
    """Names of the CUDA kernels launched inside the block (CUPTI activity records through torch.profiler)."""

    def __enter__(self):
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        self._p = profile(activities=[ProfilerActivity.CUDA])
        self._p.__enter__()
        return self

    def __exit__(self, *exc):
        self._p.__exit__(*exc)
        self.names = []
        if exc[0] is None:
            try:
                self.names = [e.name() for e in self._p.profiler.kineto_results.events()]
            except AttributeError:
                pass
            self.names += [e.name for e in self._p.events()]
        return False


def check_kernel(case, launches, expected):
    """Records the case for the coverage test and asserts the dispatch.  Call after the parity asserts: when the
    profiler records no kernel at all on this machine only the selection check is skipped."""
    got = emit_kernels(launches.names)
    OBSERVED[case] = got
    EXPECTED[case] = expected
    if not launches.names:
        pytest.skip("torch.profiler recorded no CUDA kernel here: emit kernel selection not checked (parity passed)")
    PROFILER_SAW_KERNELS.append(case)
    assert len(got) == 1, (case, sorted(got))
    if expected is not None:
        assert got == {expected}, (case, sorted(got), expected)


# ------------------------------------------------------------------------------------------------------------ inputs
def unique_keys(rng, n, klen):
    keys = rng.integers(0, 256, size=(n, klen), dtype=np.uint8)
    u = min(klen, 7)
    ids = np.unique(rng.integers(0, 1 << (8 * u), size=2 * n + 16, dtype=np.int64))
    assert ids.size >= n
    ids = rng.permutation(ids)[:n]
    keys[:, klen - u:] = ids.astype(">u8").view(np.uint8).reshape(n, 8)[:, 8 - u:]
    return keys


def records_unique(rng, n, klen, vlen):
    return unique_keys(rng, n, klen), rng.integers(0, 256, size=(n, vlen), dtype=np.uint8)


def records_repeated(rng, n, klen, vlen):
    """keys drawn from n/6 distinct ones, value = f(key): tie order cannot matter"""
    m = max(1, n // 6)
    pool_k, pool_v = records_unique(rng, m, klen, vlen)
    idx = rng.integers(0, m, size=n)
    return pool_k[idx], pool_v[idx]


def pack(keys, vals):
    return np.ascontiguousarray(np.concatenate([keys, vals], axis=1)).reshape(-1)


def n_for(r, parts, stride, factor=1.6):
    """at least three full tiles and a partial one in every partition (hash partitioning is uneven: factor)"""
    return max(8, min(int(parts * (3 * r + r // 2 + 1) * factor), MAX_BYTES // stride))


def _records_per_partition(index, rs):
    # fixed framing, no repeats: partLength = 4 (header) + records + 2 (EOF) + 4 (checksum)
    return [(int(part) - 10) // rs if part else 0 for _, _, part in index]


def _sid(shape):
    return "%dx%d" % shape


# ---------------------------------------------------------------------------------------------------- A: map side
@pytest.mark.parametrize("P", [1, 3])
@pytest.mark.parametrize("shape", MATRIX, ids=_sid)
def test_map_side_unique_keys(shape, P):
    """Unique keys, RLE auto (off): the fixed-framing emit.  Enough tiles that the persistent CTAs of the pipelined
    kernels walk several tiles each."""
    klen, vlen = shape
    stride, rs = klen + vlen, rec_size(klen, vlen)
    r = recs_per_tile(klen, vlen, True)
    n = max(n_for(r, P, stride), min(1200 * r, MAX_BYTES // stride))
    rng = np.random.default_rng(klen * 100003 + vlen * 7 + P)
    kv = pack(*records_unique(rng, n, klen, vlen))
    exp = O.pipelined_sort_fixed(O.sorter_conf(P), kv, klen, vlen)
    assert not exp["rle_used"]
    with _Launches() as la:
        with T.GpuSorter(P, fixed=shape) as s:
            s.collect_fixed(kv)
            out, index_bytes, index, st = s.flush_to_memory()
    assert out.size == len(exp["file_out"])
    assert np.array_equal(out, np.frombuffer(exp["file_out"], dtype=np.uint8)), "file.out differs from the oracle"
    assert index_bytes == exp["index_out"]
    assert np.array_equal(index, exp["index"])
    assert st["output_records"] == n and not st["rle_used"]
    assert min(_records_per_partition(exp["index"], rs)) >= 3 * r + 1
    check_kernel(("A-unique", shape, P), la, expected_emit_kernel(klen, vlen, True))


@pytest.mark.parametrize("P", [1, 3])
@pytest.mark.parametrize("shape", MATRIX, ids=_sid)
def test_map_side_repeated_keys_rle_on(shape, P):
    """Repeated keys with RLE on: records after the first of a key are written as REPEAT_KEY, so the framing is not
    constant and the variable-framing kernel takes the tile."""
    klen, vlen = shape
    stride = klen + vlen
    n = n_for(recs_per_tile(klen, vlen, True), P, stride)
    rng = np.random.default_rng(klen * 100019 + vlen * 11 + P)
    kv = pack(*records_repeated(rng, n, klen, vlen))
    exp = O.pipelined_sort_fixed(O.sorter_conf(P, rle_policy=T.RLE_ON), kv, klen, vlen)
    assert exp["rle_used"]
    with _Launches() as la:
        with T.GpuSorter(P, fixed=shape, rle_policy=T.RLE_ON) as s:
            s.collect_fixed(kv)
            out, index_bytes, index, st = s.flush_to_memory()
    assert np.array_equal(out, np.frombuffer(exp["file_out"], dtype=np.uint8)), "file.out differs from the oracle"
    assert index_bytes == exp["index_out"]
    assert np.array_equal(index, exp["index"])
    assert st["rle_used"] and st["adjacent_equal_keys"] > 0
    check_kernel(("A-rle", shape, P), la, expected_emit_kernel(klen, vlen, True, fixed_emit=False))


# ---------------------------------------------------------------------------------------- B: map side, device input
def _device_sort(kv, shape, P, offset):
    """kv copied into a tensor at byte `offset`, its last record ending at the end of the tensor"""
    import torch
    klen, vlen = shape
    n = kv.size // (klen + vlen)
    buf = torch.zeros(offset + kv.size, dtype=torch.uint8, device="cuda")
    buf[offset:] = torch.from_numpy(kv).cuda()
    cap = n * rec_size(klen, vlen) + P * 64 + 4096
    d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    with T.GpuSorter(P, fixed=shape) as s:
        with _Launches() as la:
            out_len, index, st = s.sort_device_fixed(buf.data_ptr() + offset, n, d_out.data_ptr(), cap)
            torch.cuda.synchronize()
    return d_out[:out_len].cpu().numpy(), index, st, la


@pytest.mark.parametrize("offset", [16, 48])
@pytest.mark.parametrize("shape", [s for s in MATRIX if s in ((8, 8), (16, 64), (16, 2032), (16, 32752), (10, 7), (200, 57))], ids=_sid)
def test_map_side_device_input_at_an_offset(shape, offset):
    """sort_device_fixed over records that start inside a larger buffer and end exactly at its end: no load may reach
    past the caller's bytes, and the result equals the oracle's."""
    klen, vlen = shape
    P = 3
    n = n_for(recs_per_tile(klen, vlen, True), P, klen + vlen)
    rng = np.random.default_rng(klen * 31 + vlen + offset)
    kv = pack(*records_unique(rng, n, klen, vlen))
    exp = O.pipelined_sort_fixed(O.sorter_conf(P), kv, klen, vlen)
    out, index, st, la = _device_sort(kv, shape, P, offset)
    assert np.array_equal(out, np.frombuffer(exp["file_out"], dtype=np.uint8)), "file.out differs from the oracle"
    assert np.array_equal(index, exp["index"])
    check_kernel(("B-device+%d" % offset, shape, P), la, expected_emit_kernel(klen, vlen, True))


@pytest.mark.parametrize("offset", [1, 3, 8, 15])
def test_map_side_device_input_must_be_16_byte_aligned(offset):
    """tezgpu_sorter_sort_device_fixed documents 16-byte aligned input (INTEGRATION.md 5) and refuses anything else
    with TEZGPU_E_INVALID rather than reading it."""
    import torch
    kv = pack(*records_unique(np.random.default_rng(offset), 100, 16, 64))
    buf = torch.zeros(offset + kv.size, dtype=torch.uint8, device="cuda")
    buf[offset:] = torch.from_numpy(kv).cuda()
    d_out = torch.empty(1 << 16, dtype=torch.uint8, device="cuda")
    with T.GpuSorter(2, fixed=(16, 64)) as s:
        with pytest.raises(IOError, match="16-byte aligned") as ei:
            s.sort_device_fixed(buf.data_ptr() + offset, 100, d_out.data_ptr(), d_out.numel())
    assert ei.value.code == T.E_INVALID


# ------------------------------------------------------------------------------------------- C: reduce side, run table
def sorted_segments(rng, keys, vals, nseg, min_per_seg=1):
    """splits the records over nseg plain (no RLE) IFile segments, each sorted by key bytes"""
    n = keys.shape[0]
    assert n >= nseg * min_per_seg
    owner = np.concatenate([np.repeat(np.arange(nseg), min_per_seg), rng.integers(0, nseg, size=n - nseg * min_per_seg)])
    owner = rng.permutation(owner)
    segs = []
    for g in range(nseg):
        rows = np.nonzero(owner == g)[0]
        recs = sorted((keys[i].tobytes(), vals[i].tobytes()) for i in rows)
        segs.append(O.write_ifile(recs, rle=False)[0])
    return segs


EMPTY_SEGMENT = None


def _empty():
    global EMPTY_SEGMENT
    if EMPTY_SEGMENT is None:
        EMPTY_SEGMENT = O.write_ifile([], rle=False)[0]
    return EMPTY_SEGMENT


def _merge_n(shape, parts=1):
    klen, vlen = shape
    return n_for(recs_per_tile(klen, vlen, False), parts, klen + vlen, factor=1.0)


def _reduce_segments(shape, seed, nseg):
    klen, vlen = shape
    rng = np.random.default_rng(seed)
    n = _merge_n(shape)
    keys, vals = records_unique(rng, max(n, nseg), klen, vlen)
    return sorted_segments(rng, keys, vals, nseg), rng


@pytest.mark.parametrize("mode", ["header", "no_header", "device"])
@pytest.mark.parametrize("shape", MATRIX, ids=_sid)
def test_reduce_side_run_table(shape, mode):
    """Plain segments of one declared shape (and an empty one) are merged with their records addressed in place.
    no_header: in-memory segments (body + checksum); device: segments in one device buffer starting at every address
    mod 16, used where they lie."""
    klen, vlen = shape
    nseg = 15 if mode == "device" else 3
    segs, rng = _reduce_segments(shape, klen * 7919 + vlen * 13 + len(mode), nseg)
    segs = segs[:1] + [_empty()] + segs[1:]
    exp = O.merge(segs, O.CMP_BYTES, factor=100)
    n = len(exp["records"])
    keep = None
    if mode == "header":
        m = T.GpuMerger(segs, comparator=T.CMP_BYTES, fixed=shape)
    elif mode == "no_header":
        m = T.GpuMerger([s[4:] for s in segs], comparator=T.CMP_BYTES, has_header=False, fixed=shape)
    else:
        import torch
        residues = rng.permutation(16)                      # segment i starts at an address = residues[i] mod 16
        starts, pos = [], 0
        for i, s in enumerate(segs):
            pos += (int(residues[i]) - pos) % 16 + 16
            starts.append(pos)
            pos += len(s)
        keep = torch.zeros(pos + 16, dtype=torch.uint8, device="cuda")
        host = np.zeros(pos + 16, dtype=np.uint8)
        for a, s in zip(starts, segs):
            host[a:a + len(s)] = np.frombuffer(s, dtype=np.uint8)
        keep.copy_(torch.from_numpy(host))
        base = keep.data_ptr()
        assert base % 16 == 0 and sorted((base + a) % 16 for a in starts) == list(range(16))
        m = T.GpuMerger([(base + a, len(s)) for a, s in zip(starts, segs)], comparator=T.CMP_BYTES, device_ptrs=True,
                        fixed=shape)
    with m:
        assert m.parse_info()[0] == 0, "run-table mode was not used"
        assert m.counts()[0] == n
        with _Launches() as la:
            seg, raw, part, st = m.write_ifile()
    del keep
    assert part == len(exp["ifile"]) and seg == exp["ifile"], "merged IFile differs from the oracle"
    check_kernel(("C-" + mode, shape, 1), la, expected_emit_kernel(klen, vlen, False))


@pytest.mark.parametrize("shape", MATRIX, ids=_sid)
def test_reduce_side_run_table_partitions(shape):
    """Batched reduce side: four partitions, partition 0 spread over 40 runs (more than the 32 the runs kernel plans per
    warp), the others over three runs and an empty one; every partition equals its own TezMerger merge."""
    import torch
    klen, vlen = shape
    P = 4
    rng = np.random.default_rng(klen * 104729 + vlen)
    nsegs = [40] + [3] * (P - 1)
    counts = [max(_merge_n(shape), nseg) for nseg in nsegs]
    keys, vals = records_unique(rng, sum(counts), klen, vlen)      # no key in two partitions
    segs, parts = [], []
    for p in range(P):
        a = sum(counts[:p])
        mine = sorted_segments(rng, keys[a:a + counts[p]], vals[a:a + counts[p]], nsegs[p])
        if p:
            mine.insert(1, _empty())
        segs += mine
        parts += [p] * len(mine)
    order = rng.permutation(len(segs))      # the merger groups the segments by partition itself
    segs, parts = [segs[i] for i in order], [parts[i] for i in order]
    with T.GpuMerger(segs, comparator=T.CMP_BYTES, partitions=parts, num_partitions=P, fixed=shape) as m:
        assert m.parse_info()[0] == 0, "run-table mode was not used"
        cap = m.output_bound()
        d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
        with _Launches() as la:
            nbytes, index, st = m.write_partitions_device(d_out.data_ptr(), cap)
            torch.cuda.synchronize()
        out = d_out[:nbytes].cpu().numpy().tobytes()
    off = 0
    for p in range(P):
        exp = O.merge([s for s, q in zip(segs, parts) if q == p], O.CMP_BYTES, factor=100)["ifile"]
        start, raw, part = (int(x) for x in index[p])
        assert start == off and part == len(exp)
        assert out[start:start + part] == exp, "partition %d differs from the oracle" % p
        off += part
    assert off == nbytes
    check_kernel(("C-partitions", shape, P), la, expected_emit_kernel(klen, vlen, False))


# ------------------------------------------------------------------------------------------- D: contradicted shapes
@pytest.mark.parametrize("case", ["every_record", "one_record"])
def test_declared_shape_contradicted_by_the_bytes(case):
    """(15, 65) records frame to the same 82 bytes as (16, 64) ones, so the segment lengths agree with the declared
    shape and only the framing bytes tell.  The merge must leave run-table mode and still equal TezMerger's."""
    rng = np.random.default_rng(3 if case == "every_record" else 4)
    segs = []
    for g in range(3):
        if case == "every_record":
            keys, vals = records_unique(rng, 700, 15, 65)
            recs = [(k.tobytes(), v.tobytes()) for k, v in zip(keys, vals)]
        else:
            keys, vals = records_unique(rng, 700, 16, 64)
            recs = [(k.tobytes(), v.tobytes()) for k, v in zip(keys, vals)]
            if g == 1:
                k, v = recs[350]
                recs[350] = (k[:15], v + k[15:])   # one (15, 65) record among (16, 64) ones
        segs.append(O.write_ifile(sorted(recs), rle=False)[0])
    segs.insert(2, _empty())
    assert all((len(s) - 10) % 82 == 0 for s in segs)
    exp = O.merge(segs, O.CMP_BYTES, factor=100)
    with T.GpuMerger(segs, comparator=T.CMP_BYTES, fixed=(16, 64)) as m:
        assert m.parse_info()[0] != 0, "a contradicted shape stayed in run-table mode"
        recs = list(m.records(batch_records=500, batch_bytes=1 << 16))
        with _Launches() as la:
            seg, raw, part, st = m.write_ifile()
    assert [(k, v) for k, v, _ in recs] == [(k, v) for k, v, _ in exp["records"]]
    assert seg == exp["ifile"], "merged IFile differs from the oracle"
    check_kernel(("D-" + case, (16, 64), 1), la, expected_emit_kernel(16, 64, False, fixed_emit=False))


# -------------------------------------------------------------------------------------------------------- coverage
def test_matrix_launched_its_emit_kernels():
    """Every kernel the dispatch table names for the cases that ran was seen; on the default path the full matrix
    reaches all five default-path kernels; under a sweep switch, that switch's kernel ran at least once."""
    if not OBSERVED:
        pytest.skip("no case of this file ran in this process")
    if not PROFILER_SAW_KERNELS:
        pytest.skip("torch.profiler recorded no CUDA kernel here: emit kernel selection not checked")
    seen = set().union(*OBSERVED.values())
    for case in sorted(OBSERVED, key=str):
        print("%-14s %-10s P=%d  %s" % (case[0], _sid(case[1]), case[2], ", ".join(sorted(OBSERVED[case]))))
    expected = {k for k in EXPECTED.values() if k is not None}
    assert expected <= seen, sorted(expected - seen)
    if not ACTIVE_SWITCHES:
        static = {expected_emit_kernel(k, v, a) for k, v in SHAPES for a in (True, False)}
        assert DEFAULT_PATH <= static, sorted(DEFAULT_PATH - static)
        if len(OBSERVED) == _cases_in_matrix():
            assert DEFAULT_PATH <= seen, sorted(DEFAULT_PATH - seen)
    for sw in ACTIVE_SWITCHES:
        assert SWITCHES[sw][1] in seen, (sw, sorted(seen))


def _cases_in_matrix():
    b = len([s for s in MATRIX if s in ((8, 8), (16, 64), (16, 2032), (16, 32752), (10, 7), (200, 57))])
    return len(MATRIX) * 2 * 2 + 2 * b + len(MATRIX) * 3 + len(MATRIX) + 2


# -------------------------------------------------------------------------------------------------------- F: sweep
@pytest.mark.skipif(bool(ACTIVE_SWITCHES), reason="already running under an emit switch")
@pytest.mark.parametrize("switch", sorted(SWITCHES))
def test_switch_sweep(switch):
    """Each emit switch, read once per process: parts A-D of this file in a child process with the switch set, over
    the reduced shape list; the child asserts the per-case kernels and that the switch's kernel ran."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
    env[switch] = SWITCHES[switch][0]
    cmd = [sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider",
           os.path.join("tests", os.path.basename(__file__)), "-k", "not test_switch_sweep"]
    r = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and " failed" not in r.stdout, r.stdout[-2000:]
