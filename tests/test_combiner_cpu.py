"""CPU: the reference sum combiner (tests/combine_ref.py) against a plain group-by, and the combiner configuration checks
of OrderedPartitionedKVOutput.start(), which run before the device is touched."""
import random

import numpy as np
import pytest

from oracle import tez_oracle as O
from tez_b200.runtime_library import INT_WRITABLE, TEXT, OrderedPartitionedKVOutput, OutputContext

import combine_ref as R

LONG_WRITABLE = "org.apache.hadoop.io.LongWritable"
MR_COMBINER = "org.apache.tez.mapreduce.combine.MRCombiner"
INT_SUM = "org.apache.hadoop.mapreduce.lib.reduce.IntSumReducer"


def _records(rng, n, distinct, kind):
    w = R.WIDTH[kind]
    words = ["k%d" % rng.randrange(distinct) for _ in range(n)]
    # values near the top of the range: the sums wrap around
    vals = [rng.choice([rng.getrandbits(8 * w), (1 << (8 * w)) - 1 - rng.getrandbits(4), rng.getrandbits(8)]) for _ in range(n)]
    return [O.text(x) for x in words], [v.to_bytes(w, "big") for v in vals]


def _pack(keys, values):
    kv = b"".join(k + v for k, v in zip(keys, values))
    lens = [len(k) + len(v) for k, v in zip(keys, values)]
    ko = np.cumsum([0] + lens[:-1]).astype(np.uint64) if keys else np.zeros(0, np.uint64)
    return (np.frombuffer(kv, np.uint8) if kv else np.zeros(0, np.uint8), ko, [len(k) for k in keys],
            [len(v) for v in values])


@pytest.mark.parametrize("kind", [R.INT_SUM, R.LONG_SUM])
@pytest.mark.parametrize("P,send_empty,given", [(1, True, False), (7, True, True), (64, True, False), (64, False, False),
                                                (300, False, True)])
def test_reference_combine_equals_group_by(kind, P, send_empty, given):
    rng = random.Random(P * 10 + kind)
    n = 3000
    keys, values = _records(rng, n, 400, kind)
    part = [rng.randrange(P) for _ in range(n)] if given else None
    pmode = O.PART_GIVEN if given else O.PART_HASH
    conf = O.sorter_conf(P, cmp_kind=O.CMP_TEXT, partitioner=pmode, send_empty=send_empty)
    spill = O.pipelined_sort(conf, *_pack(keys, values), partition=part)
    got = R.combine_file_out(spill["file_out"], spill["index"], kind)
    # the same output written from a plain group-by: keys are unique per partition, so the sort of the sums is exact
    groups = R.group_sum(keys, values, kind, part)
    gk = [k for _, k in groups]
    gv = list(groups.values())
    gp = [p for p, _ in groups] if given else None
    exp = O.pipelined_sort(O.sorter_conf(P, cmp_kind=O.CMP_TEXT, partitioner=pmode, send_empty=send_empty, rle_policy=0),
                           *_pack(gk, gv), partition=gp)
    assert got["file_out"] == exp["file_out"]
    assert got["index_out"] == exp["index_out"]
    assert (got["records_in"], got["records_out"]) == (n, len(groups))
    # read back: one record per (partition, key), summed with wrap-around
    back = {}
    for p in range(P):
        start, _, plen = got["index"][p]
        for ks, k, v in (O.read_ifile(got["file_out"][start:start + plen]) if plen else []):
            assert ks == O.NEW_KEY
            back[(p if given else 0, k)] = v
    assert back == groups
    empty = [p for p in range(P) if got["index"][p, 1] <= 6]
    assert len(empty) == sum(1 for p in range(P) if spill["index"][p, 1] <= 6)


@pytest.mark.parametrize("kind", [R.INT_SUM, R.LONG_SUM])
def test_vectorised_group_by_matches_the_plain_one(kind):
    rng = np.random.default_rng(kind)
    w = R.WIDTH[kind]
    n = 5000
    keys = rng.integers(0, 50, n).astype(np.uint8).repeat(16).reshape(n, 16)
    vals = rng.integers(0, 256, (n, w), dtype=np.uint8)
    part = rng.integers(0, 3, n).astype(np.int32)
    kv = np.concatenate([keys, vals], axis=1).ravel()
    out, gp = R.group_sum_fixed(kv, 16, w, kind, part)
    rows = out.reshape(-1, 16 + w)
    got = {(int(p), bytes(r[:16])): bytes(r[16:]) for p, r in zip(gp, rows)}
    assert got == R.group_sum([bytes(k) for k in keys], [bytes(v) for v in vals], kind, part)


def _start(tmp_path, extra):
    conf = {"tez.runtime.key.class": TEXT, "tez.runtime.value.class": INT_WRITABLE}
    conf.update(extra)
    out = OrderedPartitionedKVOutput(OutputContext(conf, str(tmp_path)), 2)
    out.initialize()
    try:
        out.start()
        return None
    except IOError as e:
        return str(e)


@pytest.mark.parametrize("new_api", [True, False])
def test_sum_reducer_with_the_wrong_value_class_is_rejected_at_start(tmp_path, new_api):
    key = "mapreduce.job.combine.class" if new_api else "mapred.combiner.class"
    err = _start(tmp_path, {"tez.runtime.combiner.class": MR_COMBINER, "mapred.mapper.new-api": new_api, key: INT_SUM,
                            "tez.runtime.value.class": LONG_WRITABLE})
    assert err is not None and "error -6" in err
    assert INT_SUM in err and INT_WRITABLE in err and LONG_WRITABLE in err
    err = _start(tmp_path, {"tez.runtime.combiner.class": MR_COMBINER, key: "org.apache.hadoop.mapred.lib.LongSumReducer",
                            "mapred.mapper.new-api": new_api})
    assert err is not None and "LongSumReducer" in err and "error -6" in err


def test_combiners_outside_the_sum_set_leave_start_as_it_was(tmp_path):
    plain = _start(tmp_path / "a", {})
    for extra in ({"tez.runtime.combiner.class": "org.example.MyCombiner"},
                  {"tez.runtime.combiner.class": MR_COMBINER, "mapreduce.job.combine.class": "org.example.MaxReducer",
                   "mapred.mapper.new-api": True},
                  # the reducer sits under the other API's key: MRCombiner would not find it
                  {"tez.runtime.combiner.class": MR_COMBINER, "mapred.combiner.class": INT_SUM, "mapred.mapper.new-api": True,
                   "tez.runtime.value.class": LONG_WRITABLE}):
        assert _start(tmp_path / "b", extra) == plain
