"""GPU: the device sum combiner (combine.cuh) byte for byte against the reference combine (tests/combine_ref.py) and the
CPU oracle -- sorter entry points, the merger's write paths and the OrderedPartitionedKVOutput plugin.  Values are random,
so every case also checks that the sum does not depend on the order of equal keys."""
import ctypes as C
import random

import numpy as np
import pytest

from oracle import tez_oracle as O
import tez_b200 as T
from tez_b200.runtime_library import (INT_WRITABLE, TEXT, InputContext, LocalOutput,
                                      OrderedGroupedKVInput, OrderedPartitionedKVOutput, OutputContext,
                                      empty_partitions_from_payload, parse_proto)

import combine_ref as R

pytestmark = pytest.mark.gpu

LONG_WRITABLE = "org.apache.hadoop.io.LongWritable"
KINDS = {R.INT_SUM: T.COMBINE_INT_SUM, R.LONG_SUM: T.COMBINE_LONG_SUM}


def _fixed_records(n, distinct, kind, seed):
    """n packed (16-byte key, random value) records over `distinct` keys (0 = every key unique)."""
    rng = np.random.default_rng(seed)
    w = R.WIDTH[kind]
    if distinct == 0:
        keys = rng.integers(0, 256, (n, 16), dtype=np.uint8)
    else:
        table = rng.integers(0, 256, (max(distinct, 1), 16), dtype=np.uint8)
        keys = table[rng.integers(0, distinct, n)]
    vals = rng.integers(0, 256, (n, w), dtype=np.uint8)
    return np.concatenate([keys, vals], axis=1).ravel()


def _expect_fixed(kv, P, kind, klen=16):
    w = R.WIDTH[kind]
    comb, _ = R.group_sum_fixed(kv, klen, w, kind)
    return O.pipelined_sort_fixed(O.sorter_conf(P, rle_policy=0), comb, klen, w), len(comb) // (klen + w)


def _check(out, index_bytes, st, info, exp, n, m, payload):
    assert bytes(out) == exp["file_out"], "combined file.out differs"
    assert index_bytes is None or index_bytes == exp["index_out"]
    assert info[:2] == (n, m)
    assert st["output_records"] == n and st["output_bytes"] == payload
    assert st["spilled_records"] == m
    assert st["output_bytes_with_overhead"] == exp["counters"]["OUTPUT_BYTES_WITH_OVERHEAD"]


def _run_fixed(kv, P, kind, entry, rle=T.RLE_AUTO):
    import torch
    w = R.WIDTH[kind]
    n = len(kv) // (16 + w)
    with T.GpuSorter(P, fixed=None if entry == "collect_batch" else (16, w), combiner=KINDS[kind], rle_policy=rle) as s:
        if entry == "collect_fixed":
            s.collect_fixed(kv)
            out, ib, _, st = s.flush_to_memory()
        elif entry == "collect_batch":
            ko = np.arange(n, dtype=np.uint32) * (16 + w)
            s.collect(kv, ko, ko + 16, np.full(n, w, np.uint32))
            out, ib, _, st = s.flush_to_memory()
        else:
            d_kv = torch.from_numpy(np.ascontiguousarray(kv)).cuda() if n else torch.empty(16, dtype=torch.uint8, device="cuda")
            cap = n * (16 + w + 12) + 10 * P + 64
            d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            ln, _, st = s.sort_device_fixed(d_kv.data_ptr(), n, d_out.data_ptr(), cap)
            out, ib = d_out[:ln].cpu().numpy(), None
        return out, ib, st, s.combine_info()


@pytest.mark.parametrize("kind", [R.INT_SUM, R.LONG_SUM])
@pytest.mark.parametrize("P", [1, 64, 1024])
@pytest.mark.parametrize("n,dup", [(0, 0), (1, 0), (10000, 0), (10000, 0.5), (10000, 0.999)])
def test_sorter_fixed_keys_small(kind, P, n, dup):
    distinct = 0 if dup == 0 else max(1, int(n * (1 - dup)))
    kv = _fixed_records(n, distinct, kind, seed=P + n)
    exp, m = _expect_fixed(kv, P, kind)
    out, ib, st, info = _run_fixed(kv, P, kind, "collect_fixed")
    _check(out, ib, st, info, exp, n, m, len(kv))


@pytest.mark.parametrize("entry", ["collect_fixed", "collect_batch", "sort_device_fixed"])
@pytest.mark.parametrize("kind,n,dup,P", [(R.LONG_SUM, 10 ** 6, 0.5, 64), (R.INT_SUM, 10 ** 6, 0.999, 1024),
                                          (R.LONG_SUM, 10 ** 6, 0, 64)])
def test_sorter_fixed_keys_entry_points(entry, kind, n, dup, P):
    distinct = 0 if dup == 0 else int(n * (1 - dup))
    kv = _fixed_records(n, distinct, kind, seed=7)
    exp, m = _expect_fixed(kv, P, kind)
    out, ib, st, info = _run_fixed(kv, P, kind, entry)
    _check(out, ib, st, info, exp, n, m, len(kv))


@pytest.mark.parametrize("kind,dup", [(R.LONG_SUM, 0.999), (R.INT_SUM, 0)])
def test_sorter_ten_million_records(kind, dup):
    n, P = 10 ** 7, 1024
    kv = _fixed_records(n, 0 if dup == 0 else int(n * (1 - dup)), kind, seed=11)
    exp, m = _expect_fixed(kv, P, kind)
    out, ib, st, info = _run_fixed(kv, P, kind, "sort_device_fixed")
    _check(out, ib, st, info, exp, n, m, len(kv))


def test_one_key_over_many_tiles_overflows_the_int_sum():
    """1.2e7 records of one key: the group crosses thousands of scan tiles and the int sum wraps many times."""
    n = 12 * 10 ** 6
    rng = np.random.default_rng(3)
    kv = np.empty((n, 20), np.uint8)
    kv[:, :16] = np.frombuffer(b"the-one-hot-key!", np.uint8)
    kv[:, 16:] = rng.integers(0, 256, (n, 4), dtype=np.uint8)
    total = int(kv[:, 16:].copy().view(">u4").astype(np.uint64).sum()) & 0xFFFFFFFF
    out, ib, st, info = _run_fixed(kv.ravel(), 1, R.INT_SUM, "collect_fixed")
    recs = O.read_ifile(bytes(out))
    assert [(k, v) for _, k, v in recs] == [(b"the-one-hot-key!", total.to_bytes(4, "big"))]
    assert info[:2] == (n, 1) and st["spilled_records"] == 1


def _var_records(cmp, n, distinct, kind, seed):
    rng = random.Random(seed)
    w = R.WIDTH[kind]
    if cmp == O.CMP_TEXT:
        pool = [O.text("w%x" % rng.getrandbits(40) * rng.randint(1, 3)) for _ in range(distinct)]
    elif cmp == O.CMP_INT:
        pool = [O.int_writable(rng.getrandbits(32)) for _ in range(distinct)]
    else:
        pool = [O.long_writable(rng.getrandbits(64)) for _ in range(distinct)]
    keys = [pool[rng.randrange(distinct)] for _ in range(n)]
    vals = [rng.getrandbits(8 * w).to_bytes(w, "big") for _ in range(n)]
    return keys, vals


def _pack(keys, values):
    kv = b"".join(k + v for k, v in zip(keys, values))
    lens = np.array([len(k) + len(v) for k, v in zip(keys, values)], np.int64)
    ko = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint32) if len(keys) else np.zeros(0, np.uint32)
    kl = np.array([len(k) for k in keys], np.uint32)
    vl = np.array([len(v) for v in values], np.uint32)
    return np.frombuffer(kv, np.uint8) if kv else np.zeros(0, np.uint8), ko, kl, vl


def _expect_var(keys, vals, P, cmp, kind, part=None):
    groups = R.group_sum(keys, vals, kind, part)
    gk, gv = [k for _, k in groups], list(groups.values())
    kv, ko, kl, vl = _pack(gk, gv)
    pm = O.PART_GIVEN if part is not None else O.PART_HASH
    return O.pipelined_sort(O.sorter_conf(P, cmp_kind=cmp, partitioner=pm, rle_policy=0), kv, ko.astype(np.uint64), kl, vl,
                            partition=[p for p, _ in groups] if part is not None else None), len(groups)


@pytest.mark.parametrize("cmp", [O.CMP_TEXT, O.CMP_INT, O.CMP_LONG])
@pytest.mark.parametrize("kind", [R.INT_SUM, R.LONG_SUM])
@pytest.mark.parametrize("P,given", [(1, False), (64, True), (1024, False)])
def test_sorter_variable_records(cmp, kind, P, given):
    n = 20000
    keys, vals = _var_records(cmp, n, 3000, kind, seed=cmp * 7 + P)
    part = None
    if given:
        rng = random.Random(P)
        part = [rng.randrange(P) for _ in range(n)]
    exp, m = _expect_var(keys, vals, P, cmp, kind, part)
    kv, ko, kl, vl = _pack(keys, vals)
    with T.GpuSorter(P, comparator=cmp, partitioner=T.PART_GIVEN if given else T.PART_HASH, combiner=KINDS[kind]) as s:
        s.collect(kv, ko, ko + kl, vl, None if part is None else np.array(part, np.int32))
        out, ib, _, st = s.flush_to_memory()
        info = s.combine_info()
    _check(out, ib, st, info, exp, n, m, int(kl.sum() + vl.sum()))


def test_rle_decision_is_taken_before_the_combine():
    n, P = 50000, 16
    keys, vals = _var_records(O.CMP_TEXT, n, 2000, R.LONG_SUM, seed=5)
    kv, ko, kl, vl = _pack(keys, vals)
    exp, m = _expect_var(keys, vals, P, O.CMP_TEXT, R.LONG_SUM)
    for rle in (T.RLE_ON, T.RLE_AUTO):
        with T.GpuSorter(P, comparator=T.CMP_TEXT, rle_policy=rle) as s:
            s.collect(kv, ko, ko + kl, vl)
            _, _, _, plain = s.flush_to_memory()
        with T.GpuSorter(P, comparator=T.CMP_TEXT, rle_policy=rle, combiner=T.COMBINE_LONG_SUM) as s:
            s.collect(kv, ko, ko + kl, vl)
            out, ib, idx, st = s.flush_to_memory()
        assert bytes(out) == exp["file_out"] and ib == exp["index_out"]
        assert st["rle_used"] == plain["rle_used"] == 1                    # 96 % duplicates: RLE on before the combine
        assert st["adjacent_equal_keys"] == plain["adjacent_equal_keys"] == n - m
        for p in range(P):
            seg = bytes(out[idx[p, 0]:idx[p, 0] + idx[p, 2]])
            assert all(ks == O.NEW_KEY for ks, _, _ in O.read_ifile(seg)) if idx[p, 2] else True


def test_error_paths():
    # a value of the wrong width fails the flush, with or without equal keys; the handle is usable after a reset
    for keys in ([O.text("a"), O.text("a"), O.text("b")], [O.text("a"), O.text("b"), O.text("c")]):
        vals = [O.int_writable(1), b"\0\0\0\0\0", O.int_writable(3)]
        kv, ko, kl, vl = _pack(keys, vals)
        with T.GpuSorter(2, comparator=T.CMP_TEXT, combiner=T.COMBINE_INT_SUM) as s:
            s.collect(kv, ko, ko + kl, vl)
            with pytest.raises(T._lib.TezGpuError, match="record 1 is not a 4-byte IntWritable") as e:
                s.flush_to_memory()
            assert e.value.code == T.E_INVALID
            s.reset()
            vals[1] = O.int_writable(2)
            kv, ko, kl, vl = _pack(keys, vals)
            s.collect(kv, ko, ko + kl, vl)
            out, _, _, st = s.flush_to_memory()
            assert st["spilled_records"] == len(set(keys))
    with T.GpuSorter(4, unordered=True) as s:
        with pytest.raises(T._lib.TezGpuError) as e:
            s.set_combiner(T.COMBINE_LONG_SUM)
        assert e.value.code == T.E_UNSUPPORTED
    with T.GpuSorter(4, fixed=(16, 8)) as s:
        with pytest.raises(T._lib.TezGpuError) as e:
            s.set_combiner(T.COMBINE_INT_SUM)
        assert e.value.code == T.E_INVALID
        s.set_combiner(T.COMBINE_LONG_SUM)
        s.collect_fixed(_fixed_records(10, 3, R.LONG_SUM, 1))
        with pytest.raises(T._lib.TezGpuError) as e:
            s.set_combiner(T.COMBINE_NONE)                                   # records already collected
        assert e.value.code == T.E_STATE


def _spills(keys, vals, P, cmp, nspill, rle):
    """nspill sorted spills (uncombined, rle as given) -> [(segment bytes, partition)]"""
    segs = []
    step = (len(keys) + nspill - 1) // nspill
    for a in range(0, len(keys), step):
        kv, ko, kl, vl = _pack(keys[a:a + step], vals[a:a + step])
        with T.GpuSorter(P, comparator=cmp, rle_policy=rle) as s:
            s.collect(kv, ko, ko + kl, vl)
            out, _, idx, st = s.flush_to_memory()
        assert st["rle_used"] == (rle == T.RLE_ON)
        for p in range(P):
            if idx[p, 1] > 6:
                segs.append((bytes(out[idx[p, 0]:idx[p, 0] + idx[p, 2]]), p))
    return segs


@pytest.mark.parametrize("rle", [T.RLE_ON, T.RLE_OFF])
@pytest.mark.parametrize("kind", [R.INT_SUM, R.LONG_SUM])
def test_merger_combines_its_writes(tmp_path, rle, kind):
    import torch
    n, P = 40000, 8
    keys, vals = _var_records(O.CMP_TEXT, n, 1500, kind, seed=kind + rle)
    segs = _spills(keys, vals, P, O.CMP_TEXT, 4, rle)
    exp, m = _expect_var(keys, vals, P, O.CMP_TEXT, kind)
    got = []
    for check_same in (True, False):
        with T.GpuMerger([s for s, _ in segs], comparator=T.CMP_TEXT, partitions=[p for _, p in segs], num_partitions=P) as mg:
            mg.set_check_for_same_keys(check_same)
            mg.set_combiner(KINDS[kind])
            cap = mg.output_bound()
            d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
            ln, idx, st = mg.write_partitions_device(d_out.data_ptr(), cap, rle=True)
            assert d_out[:ln].cpu().numpy().tobytes() == exp["file_out"]
            assert np.array_equal(idx, exp["index"])
            assert mg.combine_info()[:2] == (n, m) and st["spilled_records"] == m
            # the file variant (PipelinedSorter's final merge)
            f = str(tmp_path / "file.out")
            ix = np.zeros((P, 3), np.int64)
            T._lib.check(mg.L.tezgpu_merge_write_partitions(mg.h, f.encode(), (f + ".index").encode(), 1 if rle else 0,
                                                             ix.ctypes.data, C.byref(T._lib.Stats())))
            got.append(open(f, "rb").read())
            assert open(f + ".index", "rb").read() == exp["index_out"]
            # the iterator stays the uncombined TezRawKeyValueIterator stream
            assert sum(1 for _ in mg.records()) == n
    assert got[0] == got[1] == exp["file_out"]
    # one partition through write_ifile
    mine = [i for i in range(n) if O.partition_of(O.CMP_TEXT, keys[i], P) == 3]
    k3, v3 = [keys[i] for i in mine], [vals[i] for i in mine]
    segs1 = _spills(k3, v3, 1, O.CMP_TEXT, 3, rle)
    exp1, m1 = _expect_var(k3, v3, 1, O.CMP_TEXT, kind)
    with T.GpuMerger([s for s, _ in segs1], comparator=T.CMP_TEXT) as mg:
        mg.set_combiner(KINDS[kind])
        seg, raw, part, st = mg.write_ifile(rle=bool(rle))
        assert seg == exp1["file_out"] and raw == exp1["index"][0, 1]
        assert mg.combine_info()[:2] == (len(k3), m1)


def _run_output(tmp, conf, records, P, uid="attempt_1_0001_1_00_000000_0_10001"):
    out = OrderedPartitionedKVOutput(OutputContext(conf, str(tmp), unique_identifier=uid, total_memory_available_to_task=1 << 30), P)
    out.initialize()
    out.start()
    w = out.getWriter()
    for k, v in records:
        w.write(k, v)
    return out, out.close()


def _word_records(n, distinct, seed, width=8):
    rng = random.Random(seed)
    return [(O.text("word%05d" % rng.randrange(distinct)), rng.getrandbits(8 * width).to_bytes(width, "big")) for _ in range(n)]


LONG_SUM_CONF = {"tez.runtime.key.class": TEXT, "tez.runtime.value.class": LONG_WRITABLE,
                 "tez.runtime.combiner.class": "org.apache.tez.mapreduce.combine.MRCombiner", "mapred.mapper.new-api": True,
                 "mapreduce.job.combine.class": "org.apache.hadoop.mapreduce.lib.reduce.LongSumReducer",
                 "tez.runtime.io.sort.mb": 1}


@pytest.mark.parametrize("sorter", ["PIPELINED", "LEGACY"])
def test_plugin_combines_spills_and_the_final_merge(tmp_path, sorter):
    # 18-byte records (10-byte Text key, 8-byte value): 4.5 MB through the 1 MB sort buffer = at least 4 spills
    n, P = 250000, 8
    recs = _word_records(n, 20000, seed=1)
    conf = dict(LONG_SUM_CONF, **{"tez.runtime.sorter.class": sorter})
    out, events = _run_output(tmp_path, conf, recs, P)
    assert out.num_spills >= 3
    exp, m = _expect_var([k for k, _ in recs], [v for _, v in recs], P, O.CMP_TEXT, R.LONG_SUM)
    assert open(out.final_output_file, "rb").read() == exp["file_out"]
    assert open(out.final_index_file, "rb").read() == exp["index_out"]
    cin, cout = out.counter("COMBINE_INPUT_RECORDS"), out.counter("COMBINE_OUTPUT_RECORDS")
    assert n < cin < 2 * n and m < cout < n
    assert cin - n == cout - m                          # the final merge combines what the spills wrote
    assert out.counter("SPILLED_RECORDS") == cout       # every record the writers counted came out of a combine
    assert out.counter("OUTPUT_RECORDS") == n and out.counter("OUTPUT_BYTES") == sum(len(k) + len(v) for k, v in recs)
    assert out.counter("OUTPUT_BYTES_PHYSICAL") == len(exp["file_out"])
    vm = parse_proto(events[0].payload)
    assert vm[4][0] == n


def _totals(recs):
    t = {}
    for k, v in recs:
        t[k] = (t.get(k, 0) + int.from_bytes(v, "big")) & ((1 << 64) - 1)
    return t


def _read_back(tmp, conf, files, P, spill_ids=None):
    got = {}
    for p in range(P):
        inp = OrderedGroupedKVInput(InputContext(conf, str(tmp / ("r%d" % p))), 1)
        inp.initialize()
        inp.start()
        if spill_ids is None:
            inp.handleEvents([LocalOutput(0, files[0], files[0] + ".index", p)])
        else:
            inp.handleEvents([LocalOutput(0, f, f + ".index", p, spill_id=s, last_event=(s == len(files) - 1))
                              for s, f in zip(spill_ids, files)])
        r = inp.getReader()
        while r.next():
            k = r.getCurrentKey()
            assert k not in got
            got[k] = sum(int.from_bytes(v, "big") for v in r.getCurrentValues()) & ((1 << 64) - 1)
    return got


def test_plugin_below_min_spills_and_pipelined_shuffle(tmp_path):
    # 18-byte records: 4.5 MB through the 1 MB sort buffer = at least 4 spills
    n, P = 250000, 4
    recs = _word_records(n, 5000, seed=2)
    totals = _totals(recs)
    # min.spills above the spill count: spills combine, the final merge does not
    conf = dict(LONG_SUM_CONF, **{"tez.runtime.combine.min.spills": 1000})
    out, _ = _run_output(tmp_path / "a", conf, recs, P)
    assert out.num_spills >= 3
    assert out.counter("COMBINE_INPUT_RECORDS") == n
    spilled = out.counter("COMBINE_OUTPUT_RECORDS")
    assert out.counter("SPILLED_RECORDS") == 2 * spilled
    assert _read_back(tmp_path / "a", conf, [out.final_output_file], P) == totals
    # pipelined shuffle: no final merge, every spill combined and sent as it is
    conf = dict(LONG_SUM_CONF, **{"tez.runtime.enable.final-merge.in.output": False})
    out, events = _run_output(tmp_path / "b", conf, recs, P)
    S = out.num_spills
    assert S >= 3 and out.counter("COMBINE_INPUT_RECORDS") == n
    assert out.counter("SPILLED_RECORDS") == out.counter("COMBINE_OUTPUT_RECORDS")
    dms = [e for e in events if e.type == "CompositeDataMovementEvent"]
    assert [parse_proto(e.payload)[9][0] for e in dms] == list(range(S))
    uid = out.context.unique_identifier
    files = [str(tmp_path / "b" / "output" / ("%s_%d" % (uid, s)) / "file.out") for s in range(S)]
    assert _read_back(tmp_path / "b", conf, files, P, spill_ids=list(range(S))) == totals


def test_ordered_word_count_with_a_combiner_on_the_first_edge(tmp_path):
    """test_ordered_word_count_two_edges with IntSumReducer combining the tokenizer outputs: same known answer, and the
    summation tasks read one record per (producer, word)."""
    words = []
    for i in range(1, 11):
        words += ["a_%d" % i] * (22 - 2 * i)
    random.Random(3).shuffle(words)
    P = 4
    conf1 = {"tez.runtime.key.class": TEXT, "tez.runtime.value.class": INT_WRITABLE,
             "tez.runtime.combiner.class": "org.apache.tez.mapreduce.combine.MRCombiner",
             "mapred.combiner.class": "org.apache.hadoop.mapreduce.lib.reduce.IntSumReducer"}
    producers = []
    pairs = 0
    for t in range(3):
        mine = words[t::3]
        pairs += len(set(mine))
        producers.append(_run_output(tmp_path / ("t%d" % t), conf1, [(O.text(w), O.int_writable(1)) for w in mine], P,
                                     uid="attempt_1_0001_1_00_%06d_0_10001" % t))
        assert producers[-1][0].counter("COMBINE_OUTPUT_RECORDS") == len(set(mine))
    counts, read = {}, 0
    for p in range(P):
        inp = OrderedGroupedKVInput(InputContext(conf1, str(tmp_path / ("s%d" % p))), len(producers))
        inp.initialize()
        inp.start()
        inp.handleEvents([LocalOutput(i, o.final_output_file, o.final_index_file, p,
                                      empty=p in empty_partitions_from_payload(ev[-1].payload, P))
                          for i, (o, ev) in enumerate(producers)])
        r = inp.getReader()
        while r.next():
            counts[r.getCurrentKey()[1:].decode()] = sum(int.from_bytes(v, "big") for v in r.getCurrentValues())
        read += inp.counter("REDUCE_INPUT_RECORDS")
    assert counts == {"a_%d" % i: 22 - 2 * i for i in range(1, 11)}
    assert read == pairs
