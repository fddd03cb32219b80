"""Reference of the sum combiners, for the combiner tests.

Restates runCombineProcessor (SORT/PipelinedSorter.java:601-609) -> MRCombiner -> ValuesIterator grouping
(RL/common/ValuesIterator.java:177-201) -> IntSumReducer / LongSumReducer -> IFile.Writer.append (SORT/IFile.java:443-473)
on top of the CPU oracle's IFile reader and writer.  The reducers are not part of the Tez sources: they are restated from
Hadoop's published definition (the sum of the group's values, written as the group's key and one IntWritable /
LongWritable; Java int / long arithmetic wraps around).

Sums do not depend on the order of their terms, so combining the output of one sort of all records equals what a
combining spill, or a combining final merge over any number of spills, writes.
"""
import numpy as np

from oracle import tez_oracle as O

INT_SUM, LONG_SUM = 1, 2
WIDTH = {INT_SUM: 4, LONG_SUM: 8}


def sum_value(values, kind):
    """The reducer's output value for one group: big-endian, wrapped to the value width."""
    w = WIDTH[kind]
    return (sum(int.from_bytes(v, "big") for v in values) & ((1 << (8 * w)) - 1)).to_bytes(w, "big")


def combine_segment(seg, kind):
    """One sorted IFile segment (with its 'TIF' header) -> (combined segment, rawLength, partLength, records in, out)."""
    recs = O.read_ifile(seg)
    groups = []
    for _, k, v in recs:
        # every supported comparator calls keys equal only when their bytes are equal
        if groups and groups[-1][0] == k:
            groups[-1][1].append(v)
        else:
            groups.append((k, [v]))
    out, raw, part = O.write_ifile([(k, sum_value(vs, kind)) for k, vs in groups], rle=False)
    return out, raw, part, len(recs), len(groups)


def combine_file_out(file_out, index, kind):
    """A spill's file.out + index (P x 3: start, rawLength, partLength) -> dict(file_out, index, index_out, records_in,
    records_out).  Partitions without records keep their bytes and index entry as written (empty or absent)."""
    index = np.asarray(index, dtype=np.int64).reshape(-1, 3)
    out = bytearray()
    new_index = np.zeros_like(index)
    rin = rout = 0
    for p, (start, raw, part) in enumerate(index):
        seg = bytes(file_out[start:start + part])
        if part and O.read_ifile(seg):
            seg, raw, part, a, b = combine_segment(seg, kind)
            rin += a
            rout += b
        new_index[p] = (len(out), raw, part)
        out += seg
    return dict(file_out=bytes(out), index=new_index, index_out=O.spill_record_bytes(new_index.ravel()),
                records_in=rin, records_out=rout)


def group_sum(keys, values, kind, partitions=None):
    """Plain group-by: ((partition, key) -> wrapped sum) over parallel lists of key / value bytes."""
    acc = {}
    for i, (k, v) in enumerate(zip(keys, values)):
        g = (0 if partitions is None else int(partitions[i]), bytes(k))
        acc[g] = acc.get(g, 0) + int.from_bytes(v, "big")
    w = WIDTH[kind]
    return {g: (s & ((1 << (8 * w)) - 1)).to_bytes(w, "big") for g, s in acc.items()}


def group_sum_fixed(kv, klen, vlen, kind, partitions=None):
    """group_sum for n packed fixed-width records, vectorised: returns (combined kv array of klen + width records,
    combined partitions or None), groups in no particular order."""
    w = WIDTH[kind]
    assert vlen == w
    rows = np.ascontiguousarray(kv, dtype=np.uint8).reshape(-1, klen + vlen)
    n = rows.shape[0]
    if n == 0:
        return np.zeros(0, np.uint8), (None if partitions is None else np.zeros(0, np.int32))
    gk = rows[:, :klen]
    if partitions is not None:
        pb = np.asarray(partitions, dtype=">i4").view(np.uint8).reshape(n, 4)
        gk = np.concatenate([pb, gk], axis=1)
    gk = np.ascontiguousarray(gk)
    void = gk.view(np.dtype((np.void, gk.shape[1]))).ravel()
    inv = np.unique(void, return_inverse=True)[1].ravel()
    vals = np.ascontiguousarray(rows[:, klen:]).view(">u4" if w == 4 else ">u8").ravel().astype(np.uint64)
    order = np.argsort(inv, kind="stable")
    si = inv[order]
    starts = np.concatenate([[0], np.flatnonzero(si[1:] != si[:-1]) + 1])
    sums = np.add.reduceat(vals[order], starts)          # uint64 arithmetic wraps like Java's long
    first = order[starts]                                 # one record of every group
    out = np.empty((len(starts), klen + w), dtype=np.uint8)
    out[:, :klen] = rows[first, :klen]
    be = (sums & np.uint64(0xFFFFFFFF)).astype(">u4") if w == 4 else sums.astype(">u8")
    out[:, klen:] = be.view(np.uint8).reshape(-1, w)
    return out.ravel(), (None if partitions is None else np.asarray(partitions, np.int32)[first])
