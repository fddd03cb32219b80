"""Plain flush against combining flush (LongSumReducer) on device-resident records, through
tezgpu_sorter_sort_device_fixed: n x (16-byte key, 8-byte LongWritable), P partitions, hash partitioner.

Key shapes: every key unique, 1e6 and 1e3 distinct keys, Zipf(1.1) over 1e7 ranks.  Per shape the two variants run
alternately in one process over the same input (warm-up, then timed steps; CUDA events on the sorter's stream around
each flush).  Before timing, the combined output of every shape is checked byte for byte against a host group-by
written by the CPU oracle, at --verify-records.  Prints one JSON line (and writes it to --out).

usage: python tools/combine_bench.py [--records 100000000] [--steps 5] [--warmup 1] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import tez_b200 as T  # noqa: E402
from oracle import tez_oracle as O  # noqa: E402

KLEN, VLEN = 16, 8


def gen(shape, n, seed, dev):
    """(n, 24) uint8 records on the device, and the key id of every record (None: every key distinct)"""
    g = torch.Generator(device=dev).manual_seed(seed)
    vals = torch.randint(0, 256, (n, VLEN), dtype=torch.uint8, device=dev, generator=g)
    if shape == "unique":
        keys, ids = torch.randint(0, 256, (n, KLEN), dtype=torch.uint8, device=dev, generator=g), None
    else:
        if shape == "zipf1.1":
            ranks = torch.arange(1, 10_000_001, dtype=torch.float64, device=dev)
            cdf = torch.cumsum(ranks.pow(-1.1), 0)
            cdf /= cdf[-1].clone()
            u = torch.rand(n, dtype=torch.float64, device=dev, generator=g)
            ids = torch.searchsorted(cdf, u).clamp_(max=len(ranks) - 1)
            nkeys = len(ranks)
        else:
            nkeys = int(float(shape.split("_")[0]))
            ids = torch.randint(0, nkeys, (n,), device=dev, generator=g)
        table = torch.randint(0, 256, (nkeys, KLEN), dtype=torch.uint8, device=dev, generator=g)
        keys = table[ids]
    return torch.cat([keys, vals], 1).contiguous(), ids


def expected(kv, ids, P):
    """host group-by (sum per key, wrapped to 64 bits) written by the CPU oracle's sorter"""
    rows = kv.cpu().numpy()
    if ids is None:
        comb = rows
    else:
        ids = ids.cpu().numpy()
        order = np.argsort(ids, kind="stable")
        si = ids[order]
        starts = np.concatenate([[0], np.flatnonzero(si[1:] != si[:-1]) + 1])
        vals = np.ascontiguousarray(rows[:, KLEN:]).view(">u8").ravel().astype(np.uint64)
        sums = np.add.reduceat(vals[order], starts)
        comb = np.empty((len(starts), KLEN + VLEN), np.uint8)
        comb[:, :KLEN] = rows[order[starts], :KLEN]
        comb[:, KLEN:] = sums.astype(">u8").view(np.uint8).reshape(-1, VLEN)
    return O.pipelined_sort_fixed(O.sorter_conf(P, rle_policy=0), comb.ravel(), KLEN, VLEN)["file_out"], comb.shape[0]


def flush(s, kv, d_out):
    st = torch.cuda.ExternalStream(s.stream())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    ln, _, stats = s.sort_device_fixed(kv.data_ptr(), kv.shape[0], d_out.data_ptr(), d_out.numel())
    e1.record(st)
    e1.synchronize()
    return e0.elapsed_time(e1), ln, stats


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    name, _, power = line.partition(",")
    return {"gpu": name.strip() or torch.cuda.get_device_name(0), "power_limit": power.strip() or "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=100_000_000)
    ap.add_argument("--partitions", type=int, default=64)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--verify-records", type=int, default=20_000_000)
    ap.add_argument("--shapes", default="unique,1e6_keys,1e3_keys,zipf1.1")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "combine_bench measures the GPU: no CUDA device"
    dev = torch.device("cuda", 0)
    P, n = a.partitions, a.records
    plain = T.GpuSorter(P, fixed=(KLEN, VLEN))
    comb = T.GpuSorter(P, fixed=(KLEN, VLEN), combiner=T.COMBINE_LONG_SUM)
    cap = max(n, a.verify_records) * (KLEN + VLEN + 12) + 10 * P + 64
    d_out = torch.empty(cap, dtype=torch.uint8, device=dev)
    res = dict(gpu_info(), records=n, partitions=P, record_bytes=KLEN + VLEN, steps=a.steps, warmup=a.warmup, shapes={})
    for si, shape in enumerate(a.shapes.split(",")):
        # correctness first, at the verification size
        kv, ids = gen(shape, a.verify_records, 100 + si, dev)
        torch.cuda.synchronize()
        _, ln, _ = flush(comb, kv, d_out)
        exp, m = expected(kv, ids, P)
        got = d_out[:ln].cpu().numpy().tobytes()
        assert got == exp, "%s: combined file.out differs from the host group-by" % shape
        assert comb.combine_info()[:2] == (a.verify_records, m)
        del kv, ids
        kv, _ = gen(shape, n, si, dev)
        torch.cuda.synchronize()
        t_plain, t_comb, t_phase = [], [], []
        for step in range(a.warmup + a.steps):
            tp, _, _ = flush(plain, kv, d_out)
            tc, _, _ = flush(comb, kv, d_out)
            cin, cout, cms = comb.combine_info()
            if step >= a.warmup:
                t_plain.append(tp)
                t_comb.append(tc)
                t_phase.append(cms)
        res["shapes"][shape] = dict(plain_flush_ms=float(np.median(t_plain)), combining_flush_ms=float(np.median(t_comb)),
                                    combine_phase_ms=float(np.median(t_phase)), records_in=cin, records_out=cout,
                                    plain_steps_ms=[round(x, 3) for x in t_plain],
                                    combining_steps_ms=[round(x, 3) for x in t_comb],
                                    verified_records=a.verify_records)
        del kv
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
