#!/usr/bin/env python
"""bench.py -- sorted-KV GB/s of the Tez shuffle sort/merge hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

N=1 workload = BASELINE config 2: 1e8 records, 16 B key / 64 B value, 64 partitions (HashPartitioner,
TezBytesComparator) -> file.out bytes bit-identical to the reference format.  A "step" is one complete pass of the
hot path over that batch (partition + sort + IFile emit with CRC); every GPU leg of the N=1 run times K steps.
--dump-outputs DIR (N=1): writes what the last timed step returned as DIR/*.npy (see dump_outputs), so that two builds
can be compared output for output; the inputs are the same seeded records in every run.
  value   : KV payload GB/s with the records already resident in HBM (device-timed, CUDA events on the library stream)
  e2e     : the same metric through the C ABI with HOST buffers (H2D of the records and D2H of file.out inside the
            timed region) -- the call a Tez task makes
  roofline: the dominant kernel (gather+emit) against the measured HBM copy bandwidth
N>1 (torchrun, one rank per GPU): BASELINE config 4 shape, weak scaling -- every rank sorts its own records into
1024 partitions, partitions are exchanged with an all-to-all over NVLink (owner(p) = p*N/P), each rank merges the
N runs of every partition it owns.
--impl reference: the CPU restatement of PipelinedSorter (oracle/, "port") timed on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

KEY_LEN, VAL_LEN = 16, 64
REC = KEY_LEN + VAL_LEN
OUT_REC = REC + 2                      # vint(16) vint(64) key value
ALGO_BYTES_PER_RECORD = REC + OUT_REC  # SURVEY 8(d): read 80 + write 82 = 162 B / record
METRIC = "sorted KV GB/s (16B key / 64B val)"


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_sample(cores, per_task):
    """Bounded sample of the same workload for the CPU arm: `cores` independent PipelinedSorter tasks.  Same bytes as
    synth.gen_c2 (tests/test_synth.py), from the oracle's C generator on all cores (the torch CPU path needs minutes)."""
    from oracle import tez_oracle as O
    n = cores * per_task
    return O.gen_c2(0, n, seed=2, threads=cores), n


def run_cpu(cores, per_task, steps, warmup, partitions):
    from oracle import tez_oracle as O
    kv, n = cpu_sample(cores, per_task)
    conf = O.sorter_conf(partitions)
    times = []
    for i in range(warmup + steps):
        secs, _ = O.bench_pipelined_fixed(conf, kv, KEY_LEN, VAL_LEN, cores)
        if i >= warmup:
            times.append(secs)
    t = sum(times) / len(times)
    return n * REC / t / 1e9, t, n


class gpu_local_cpus:
    """Pins the calling thread (and the threads it starts) to the CPUs NVML reports as local to a GPU while the pinned
    host buffers of the e2e leg are allocated (first touch decides their NUMA node) and copied, then restores the mask.
    Host memory on the far socket costs PCIe copies a hop over the inter-socket link.  Best effort: any failure
    leaves the affinity untouched."""

    def __init__(self, device_index=0):
        self.device_index, self.old, self.cpus = device_index, None, None

    def __enter__(self):
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                pr = torch.cuda.get_device_properties(self.device_index)
                h = pynvml.nvmlDeviceGetHandleByPciBusId(("%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)).encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.device_index)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, ((os.cpu_count() or 64) + 63) // 64)
            local = {64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1}
            old = os.sched_getaffinity(0)
            cpus = local & old
            if cpus and cpus != old:
                os.sched_setaffinity(0, cpus)
                self.old, self.cpus = old, cpus
        except Exception:
            self.old = None
        return self

    def __exit__(self, *a):
        if self.old is not None:
            try:
                os.sched_setaffinity(0, self.old)
            except Exception:
                pass
        return False


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def single_sorter_cpu(records, partitions, threads, repeats=3):
    """The config-2 shape itself on the host: ONE PipelinedSorter over `records` records (spans of 2^20 records sorted
    by `threads` sort threads, SpanMerger heap over the spans, one IFile writer), `repeats` runs -> GB/s of each."""
    from oracle import tez_oracle as O
    kv = O.gen_c2(0, records, seed=2, threads=min(host_cores(), 32))
    conf = O.sorter_conf(partitions, sort_threads=threads)
    out = []
    for _ in range(repeats):
        secs, _ = O.bench_pipelined_fixed(conf, kv, KEY_LEN, VAL_LEN, 1)
        out.append(round(records * REC / secs / 1e9, 4))
    return out


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = min(host_cores(), 128)
    per_task = args.cpu_records_per_task
    partitions = 64 if args.gpus == 1 else 1024
    value, secs, n = run_cpu(cores, per_task, args.steps, args.warmup, partitions)
    sample = "%d records (%d per task x %d tasks, one PipelinedSorter task per core, %d spans + SpanMerger each)" % (
        n, per_task, cores, (per_task + (1 << 20) - 1) >> 20)
    single = None
    if args.cpu_single_records > 0:
        # one sorter, as BASELINE.md describes config 2, on a bounded sample: tez.runtime.pipelined.sorter.sort.threads
        # = 2 (the default) and = cores; three repeats each (the spread is the honest error bar of this arm)
        single = {"records": args.cpu_single_records,
                  "sort_threads_2_gbs": single_sorter_cpu(args.cpu_single_records, partitions, 2),
                  "sort_threads_%d_gbs" % cores: single_sorter_cpu(args.cpu_single_records, partitions, cores)}
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(secs * 1e3, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.gpus, args.records),
        "cpu_baseline": {"value": round(value, 4), "unit": "GB/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 4), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU restatement of PipelinedSorter (oracle/tez_oracle.c), not the JVM: no JDK / Hadoop jars exist in this image; "
                "value = all host cores busy with independent sorter tasks (the most favourable use of the box for the CPU); "
                "single_sorter = ONE sorter over a bounded sample of config 2 at sort.threads 2 and = cores, three repeats",
    }
    if single:
        line["cpu_baseline"]["single_sorter"] = single
    print(json.dumps(line))
    return 0


def workload_config(gpus, records, config=4):
    if config == 5:
        return {"workload": "BASELINE config 5 shape (weak): %d records per GPU, Zipf(1.1) keys over 2^32 ids, 16B key / 4 KB value, "
                            "256 partitions, owner(p) = p*N/P, NVLink pull, per-GPU batched merge of run-length encoded segments" % records,
                "records_per_gpu": records, "partitions": 256, "parallelism": "partition-sharded x%d" % gpus,
                "l2": "inputs larger than L2, no flush needed"}
    if gpus == 1:
        return {"workload": "BASELINE config 2: %d records, 16B key / 64B value, 64 partitions, HashPartitioner, "
                            "TezBytesComparator, IFile + CRC32 out" % records,
                "records": records, "partitions": 64, "l2": "inputs (8 GB) larger than L2, no flush needed"}
    return {"workload": "BASELINE config 4 shape (weak): %d records per GPU, 1024 partitions, all-to-all by "
                        "partition owner (contiguous blocks, owner(p) = p*N/P) over NVLink, per-GPU batched k-way merge" % records,
            "records_per_gpu": records, "partitions": 1024, "parallelism": "partition-sharded x%d" % gpus,
            "l2": "inputs larger than L2, no flush needed"}


def load_traffic():
    p = os.path.join(ROOT, "profiles", "emit_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def dump_outputs(out_dir, d_out, out_len, index, chunks=2048, chunk_bytes=4096, seed=0):
    """What one sort_device_fixed call hands its caller, as float arrays (about 34 MB in all):
      index.npy                  (P, 3) float64: segment start, raw length, part length of every partition
      file_out_len.npy           (1,) float64: bytes of file.out
      segment_crc32.npy          (P,) float64: every segment's CRC32 trailer (covers all of its bytes; -1 = no segment)
      file_out_sample.npy        (chunks, chunk_bytes) float32: file.out bytes at seeded offsets
      file_out_sample_offsets.npy (chunks,) float64: those offsets
    The offsets depend only on `seed` and the output length, so equal outputs give equal files."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    out = d_out[:out_len]
    index = np.asarray(index, dtype=np.int64)
    crc = np.full(len(index), -1.0)
    has = index[:, 2] > 0
    if has.any():
        at = torch.from_numpy(index[has, 0] + index[has, 2] - 4)[:, None] + torch.arange(4)
        b = out[at.to(out.device)].cpu().numpy().astype(np.uint64)
        crc[has] = (b[:, 0] << 24) | (b[:, 1] << 16) | (b[:, 2] << 8) | b[:, 3]
    width = min(chunk_bytes, out_len)
    offs = np.sort(np.random.default_rng(seed).integers(0, out_len - width + 1, size=chunks))
    at = (torch.from_numpy(offs)[:, None] + torch.arange(width)).to(out.device)
    sample = out[at].cpu().numpy().astype(np.float32)
    for name, a in (("index", index.astype(np.float64)), ("file_out_len", np.array([out_len], dtype=np.float64)),
                    ("segment_crc32", crc), ("file_out_sample", sample),
                    ("file_out_sample_offsets", offs.astype(np.float64))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def single_gpu(args):
    import torch
    import tez_b200 as T
    from tez_b200 import synth
    n, P = args.records, 64
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    d_kv = synth.gen_c2(0, n, seed=2, device=dev)
    sorter = T.GpuSorter(P, fixed=(KEY_LEN, VAL_LEN), device=0)
    cap = n * OUT_REC + 10 * P + 4096
    d_out = torch.empty(cap, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    stream = torch.cuda.ExternalStream(sorter.stream(), device=dev)

    def step():
        return sorter.sort_device_fixed(d_kv.data_ptr(), n, d_out.data_ptr(), cap)

    for _ in range(args.warmup):
        step()
    clocks = ClockSampler(0)
    clocks.start()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    launches, emit_ms, stage_ms, sort_ms, ties_ms = 0, [], [], [], []
    for _ in range(args.steps):
        out_len, index, st = step()
        launches += st["kernel_launches"]
        emit_ms.append(st["ms_emit_kernel"])
        stage_ms.append(st["ms_stage"])
        sort_ms.append(st["ms_sort"])
        ties_ms.append(st["ms_ties"])
    ev1.record(stream)
    torch.cuda.synchronize()
    clk = clocks.stop()
    ms_step = ev0.elapsed_time(ev1) / args.steps
    value = n * REC / (ms_step * 1e-3) / 1e9
    assert out_len == n * OUT_REC + 10 * int((index[:, 1] > 0).sum())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, d_out, out_len, index)

    peak, peak_src = hbm_peak()
    emit = sum(emit_ms) / len(emit_ms)
    achieved = n * ALGO_BYTES_PER_RECORD / (emit * 1e-3) / 1e9
    traffic = load_traffic()
    roofline = {"bound": "hbm", "kernel": "k_emit_fast4<5,1> (software-pipelined gather + IFile framing + CRC32 + coalesced store)",
                "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": traffic["dram_bytes_per_launch"] if traffic else None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": n * ALGO_BYTES_PER_RECORD, "ms_per_launch": round(emit, 4)}
    pipeline = {"algorithmic_bytes_per_step": n * ALGO_BYTES_PER_RECORD,
                "achieved": round(n * ALGO_BYTES_PER_RECORD / (ms_step * 1e-3) / 1e9, 1),
                "frac": round(n * ALGO_BYTES_PER_RECORD / (ms_step * 1e-3) / 1e9 / peak, 4),
                "ms": {"stage": round(sum(stage_ms) / len(stage_ms), 4), "sort": round(sum(sort_ms) / len(sort_ms), 4),
                       "ties": round(sum(ties_ms) / len(ties_ms), 4), "emit_kernel": round(emit, 4)}}

    # ---- the N>1 pipeline at G=1 (BASELINE config 4 shape on one GPU: sort into 1024 partitions, no exchange, batched
    # device merge of the single run of every partition) so that the 1->N curve can also be read like for like: the
    # N=1 headline above is config 2 (sort only, P=64), the N>1 lines are sort + exchange + merge (P=1024).
    pipeline_g1 = None
    if not args.no_g1_pipeline:
        P4 = 1024
        s4 = T.GpuSorter(P4, fixed=(KEY_LEN, VAL_LEN), device=0)
        cap4 = n * OUT_REC + 10 * P4 + 4096
        d_out4 = torch.empty(cap4, dtype=torch.uint8, device=dev)
        d_merged = torch.empty(cap4 + (1 << 20), dtype=torch.uint8, device=dev)
        mg = [None]

        def step4():
            out_len4, index4, st4 = s4.sort_device_fixed(d_kv.data_ptr(), n, d_out4.data_ptr(), cap4)
            segs4 = [(d_out4.data_ptr() + int(index4[p, 0]), int(index4[p, 2])) for p in range(P4) if index4[p, 2]]
            parts4 = [p for p in range(P4) if index4[p, 2]]
            if mg[0] is None:
                mg[0] = T.GpuMerger(segs4, comparator=T.CMP_BYTES, device=0, device_ptrs=True, fixed=(KEY_LEN, VAL_LEN),
                                    partitions=parts4, num_partitions=P4)
            else:
                mg[0].reopen(segs4, parts4)
            mlen4, mindex4, mst4 = mg[0].write_partitions_device(d_merged.data_ptr(), d_merged.numel())
            return st4, mst4, mlen4, out_len4

        for _ in range(2):
            step4()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        k4 = args.steps
        for _ in range(k4):
            st4, mst4, mlen4, out_len4 = step4()
        torch.cuda.synchronize()
        ms4 = (time.perf_counter() - t0) / k4 * 1e3
        assert mlen4 == out_len4       # one run per partition: the merge reproduces the sorter's file.out length
        pipeline_g1 = {"workload": "config 4 shape at G=1: %d records, 1024 partitions, sort + batched merge (no exchange)" % n,
                       "ms_per_step": round(ms4, 3), "value": round(n * REC / (ms4 * 1e-3) / 1e9, 1), "unit": "GB/s",
                       "ms_sort": round(st4["ms_total"], 3), "ms_merge_emit": round(mst4["ms_emit"], 3),
                       "timing": "host clock around fully synchronised library calls, %d steps" % k4}
        mg[0].close()
        s4.close()
        del d_out4, d_merged

    # ---- e2e through the C ABI with host buffers (pinned), H2D + D2H inside the timed region.
    # Two task slots (as a node runs several map tasks per GPU): each slot is one sorter handle doing
    # collect (H2D of the step's 8 GB) -> flush (sort + D2H of the step's 8.2 GB file.out); with two slots the H2D of one
    # step overlaps the D2H of the other on the full-duplex PCIe link.  Every step still copies its own input and output.
    e2e = None
    if not args.no_e2e:
        with gpu_local_cpus(0) as numa:
            slots = 2
            h_kv = torch.empty(n * REC, dtype=torch.uint8, pin_memory=True)
            h_kv.copy_(d_kv)
            h_outs = [torch.empty(cap + 4096, dtype=torch.uint8, pin_memory=True) for _ in range(slots)]
            torch.cuda.synchronize()
            sorters = [T.GpuSorter(P, fixed=(KEY_LEN, VAL_LEN), device=0) for _ in range(slots)]
            esteps = args.steps
            out_bytes = [0] * slots

            # --e2e-direction-locks: one transfer at a time per PCIe direction (a slot's upload next to the other slot's
            # download; the link does 55.6 / 54.3 GB/s alone, 46 + 46 GB/s together: tools/pcie_probe.py).  Measured
            # SLOWER than letting the two slots run free (286 vs 240 ms per step), hence off; tools/e2e_probe.py prints
            # the timeline of both.
            class _free:
                def __enter__(self): return self
                def __exit__(self, *a): return False
            up = threading.Lock() if args.e2e_direction_locks else _free()
            down = threading.Lock() if args.e2e_direction_locks else _free()

            def e2e_worker(k, nsteps, go, uploaded):
                s2, ho = sorters[k], h_outs[k].numpy()
                go.wait()       # tasks do not start in the same instant: slot k+1 starts when slot k has uploaded its
                for i in range(nsteps):   # first input, so one slot's upload runs next to the other's download from step 0
                    s2.reset()
                    with up:
                        s2.collect_fixed(h_kv.data_ptr(), n=n)
                    if i == 0:
                        uploaded.set()
                    with down:
                        out, _, _, _ = s2.flush_to_memory(out=ho)
                    out_bytes[k] = int(len(out))

            def run_e2e(total_steps):
                ev = [threading.Event() for _ in range(slots + 1)]
                ev[0].set()
                per_slot = [total_steps // slots + (k < total_steps % slots) for k in range(slots)]
                ths = [threading.Thread(target=e2e_worker, args=(k, per_slot[k], ev[k], ev[k + 1])) for k in range(slots)]
                for t in ths:
                    t.start()
                for t in ths:
                    t.join()

            run_e2e(slots)  # warm-up: allocations, pinning
            t0 = time.perf_counter()
            run_e2e(esteps)
            torch.cuda.synchronize()
            t = (time.perf_counter() - t0) / esteps
            e2e = {"value": round(n * REC / t / 1e9, 3), "unit": "GB/s", "h2d_bytes_per_step": n * REC,
                   "d2h_bytes_per_step": out_bytes[0], "ms_per_step": round(t * 1e3, 2), "steps": esteps,
                   "task_slots": slots, "host_cpus_pinned_to_gpu_numa_node": len(numa.cpus) if numa.cpus else None,
                   "api": "tezgpu_sorter_collect_fixed + tezgpu_sorter_flush_to_memory (pinned host buffers), 2 task slots, the second one starts after the first one's first upload"}
            for s2 in sorters:
                s2.close()
            del h_kv, h_outs

    # ---- CPU baseline on this box's host cores (bounded sample)
    cores = min(host_cores(), 128)
    cval, csecs, cn = run_cpu(cores, args.cpu_records_per_task, 1, 0, P)
    cpu = {"value": round(cval, 4), "unit": "GB/s", "cores": cores, "kind": "port",
           "sample": "%d records (%d per task x %d PipelinedSorter tasks), %.2f s" % (cn, args.cpu_records_per_task, cores, csecs)}

    line = {"metric": METRIC, "value": round(value, 3), "unit": "GB/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(1, n),
            "clocks": clk, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "pipeline": pipeline,
            "config4_pipeline_g1": pipeline_g1, "cpu_baseline": cpu}
    print(json.dumps(line))
    return 0


def config1(args):
    """BASELINE config 1: OrderedWordCount (tez-examples OrderedWordCount.java:124-180), ~100 MB of synthetic text, 4
    tokenizer tasks, 4 reducers, local mode: both ordered edges through the plugin mirror (C++ host layer over the CUDA
    library, real files / indexes / counters), beside the same job through the CPU restatement of PipelinedSorter +
    TezMerger -- the configuration the reference itself runs on a CPU.  tools/owc_bench.cc drives both arms and checks
    the job's known answer."""
    import tempfile
    exe = os.path.join(ROOT, "tools", "owc_bench")
    if not os.path.exists(exe):
        import __graft_entry__
        __graft_entry__.build_tools()
    mb, toks, reds = args.c1_text_mb, 4, 4
    with tempfile.TemporaryDirectory() as wd:
        g = json.loads(subprocess.check_output([exe, "gpu", str(mb), str(toks), str(reds), wd], text=True).strip().splitlines()[-1])
        c = json.loads(subprocess.check_output([exe, "cpu", str(mb), str(toks), str(reds), wd], text=True).strip().splitlines()[-1])
    line = {"metric": METRIC.replace("(16B key / 64B val)", "(OrderedWordCount, both ordered edges)"), "value": round(g["kv_gbs"], 4),
            "unit": "GB/s", "n_gpus": 1, "steps": 1, "warmup": 1, "ms_per_step": round(g["seconds"] * 1e3, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "BASELINE config 1: OrderedWordCount, %d MB of synthetic text (Zipf(1.0) over 1000 words), %d tokenizer "
                                   "tasks, %d reducers, local mode, files + indexes + counters as Tez" % (mb, toks, reds),
                       "records": g["records"], "timing": "wall clock of the shuffle-bound part of the job (sort, spill files, merge, "
                                                          "grouping, second ordered edge), host buffers and local files inside"},
            "e2e": {"value": round(g["kv_gbs"], 4), "unit": "GB/s", "note": "the job IS the end-to-end path: records enter through "
                    "KeyValuesWriter.write and leave through KeyValuesReader"},
            "gpu_launches": None, "roofline": None,
            "parity": {"known_answer_checked_both_arms": bool(g["answer_checked"] and c["answer_checked"])},
            "cpu_baseline": {"value": round(c["kv_gbs"], 5), "unit": "GB/s", "cores": 2, "kind": "port",
                             "sample": "the whole job through the CPU restatement (PipelinedSorter with sort.threads=2, TezMerger), %.2f s" % c["seconds"]}}
    print(json.dumps(line))
    return 0


def config3(args):
    """BASELINE config 3: k-way TezMerger of sorted spill segments with variable-length Text keys on one GPU.
    Inputs: --c3-segments IFile segments of --c3-segment-mb MiB (SURVEY 8d generator: words from a 2^24-id space, length
    U[4,24], 8-byte value = f(word), every word at most once per segment), resident in HBM when the timed region starts.
    A step = tezgpu_merge_reopen (header / checksum verification, parallel parse, merge) + tezgpu_merge_write_ifile_device
    (TezMerger.writeFile with REPEAT_KEY run-length encoding, CRC32)."""
    import zlib
    import numpy as np
    import torch
    import tez_b200 as T
    from oracle import tez_oracle as O      # generator + checker + CPU arm (test infrastructure, never the product path)
    nseg, seg_bytes = args.c3_segments, args.c3_segment_mb << 20
    cores = min(host_cores(), 128)
    t0 = time.perf_counter()
    segs, nrec = O.gen_c3_segments(nseg, seg_bytes, seed=3, threads=cores)
    t_gen = time.perf_counter() - t0
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    offs, total = [], 0
    for a in segs:
        offs.append(total)
        total = (total + a.size + 15) // 16 * 16
    d_in = torch.empty(total + 64, dtype=torch.uint8, device=dev)
    for a, o in zip(segs, offs):
        d_in[o:o + a.size].copy_(torch.from_numpy(a))
    torch.cuda.synchronize()
    in_bytes = sum(a.size for a in segs)
    kv_in = in_bytes - 10 * nseg - 2 * sum(nrec)          # segment = 10 framing bytes + records of 2 vint bytes + key + value
    seg_list = [(d_in.data_ptr() + o, a.size) for a, o in zip(segs, offs)]
    m = T.GpuMerger(seg_list, comparator=T.CMP_TEXT, device=0, device_ptrs=True)
    bound = m.output_bound()
    d_out = torch.empty(bound + 64, dtype=torch.uint8, device=dev)

    def step():
        m.reopen(seg_list)
        return m.write_ifile_device(d_out.data_ptr(), bound)

    for _ in range(max(1, args.warmup)):
        raw, part, st = step()
    clocks = ClockSampler(0)
    clocks.start()
    torch.cuda.synchronize()
    times, launches = [], 0
    for _ in range(args.steps):
        t0 = time.perf_counter()
        raw, part, st = step()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        launches += st["kernel_launches"]
    clk = clocks.stop()
    ms_step = sum(times) / len(times) * 1e3
    records, kv_bytes = m.counts()
    parse_mode, parse_rounds = m.parse_info()
    assert records == sum(nrec) and kv_bytes == kv_in
    value = kv_bytes / (ms_step * 1e-3) / 1e9
    peak, peak_src = hbm_peak()
    algo = in_bytes + part
    # ---- parity, outside the timed region: CRC32 trailer with zlib over the whole output; byte-exact against the CPU
    # oracle's TezMerger on a bounded sample of the same segments (which is also the CPU arm)
    out = d_out[:part].cpu().numpy()
    crc_ok = int.from_bytes(out[-4:].tobytes(), "big") == zlib.crc32(out[4:-4])
    sample = max(2, min(nseg, args.c3_cpu_segments))
    exp, n_cpu, secs = O.merge_ifile(segs[:sample], O.CMP_TEXT, factor=100)
    m.reopen(seg_list[:sample])
    raw_s, part_s, _ = m.write_ifile_device(d_out.data_ptr(), bound)
    got = d_out[:part_s].cpu().numpy()
    bit_exact = bool(part_s == exp.size and np.array_equal(got, exp))
    kv_sample = sum(a.size for a in segs[:sample]) - 10 * sample - 2 * sum(nrec[:sample])
    cpu = {"value": round(kv_sample / secs / 1e9, 4), "unit": "GB/s", "cores": 1, "kind": "port",
           "sample": "%d of the %d segments (%d records) through the TezMerger restatement, factor 100, one thread "
                     "(a TezMerger merge is single-threaded), %.1f s" % (sample, nseg, n_cpu, secs)}
    line = {"metric": METRIC.replace("(16B key / 64B val)", "(k-way merge, Text keys)"), "value": round(value, 3), "unit": "GB/s",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "BASELINE config 3: k-way TezMerger of %d sorted IFile segments of %d MiB, Text keys U[4,24] from a "
                                   "2^24-word space, 8 B values, REPEAT_KEY output" % (nseg, args.c3_segment_mb),
                       "segments": nseg, "records": records, "input_bytes": in_bytes, "output_bytes": int(part),
                       "l2": "inputs larger than L2, no flush needed", "timing": "host clock around fully synchronised library calls",
                       "generation_s": round(t_gen, 1),
                       "parser": {1: "window parser (guess / evaluate / chase), %d windows walked by hand" % parse_rounds, 2: "sequential walker (window parser gave up)"}.get(parse_mode, str(parse_mode))},
            "clocks": clk, "e2e": None, "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "whole merge step (parse + sort + emit)", "achieved": round(algo / (ms_step * 1e-3) / 1e9, 1),
                         "peak": peak, "unit": "GB/s", "frac": round(algo / (ms_step * 1e-3) / 1e9 / peak, 4), "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": int(algo),
                         "note": "algorithmic bytes = segment bytes read + merged bytes written (SURVEY 8d)"},
            "phases_ms": {k: round(v, 3) for k, v in st.items() if k.startswith("ms_")},
            "parity": {"crc32_of_full_output_matches_zlib": bool(crc_ok), "bit_exact_vs_oracle_on_sample": bit_exact,
                       "sample_segments": sample},
            "cpu_baseline": cpu}
    print(json.dumps(line))
    assert crc_ok and bit_exact, "config 3 output differs from the checker"
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of every GPU leg")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--records", type=int, default=None,
                    help="records per GPU (default: 1e8 at N=1 = BASELINE config 2; 1.25e8 at N>1 = config 4's 1e9 over 8 GPUs)")
    ap.add_argument("--cpu-records-per-task", type=int, default=1_500_000,
                    help="CPU arm: records per PipelinedSorter task (> 2^20 so that every task has two spans and its SpanMerger runs)")
    ap.add_argument("--cpu-single-records", type=int, default=10_000_000,
                    help="reference arm: records of the single-sorter sample (0 = skip)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-direction-locks", action="store_true", help="e2e leg: serialise the task slots per PCIe direction")
    ap.add_argument("--no-g1-pipeline", action="store_true")
    ap.add_argument("--config", type=int, default=2,
                    help="2 (default, the driver's line), 1 (OrderedWordCount through the plugin mirror), 3 (k-way merge) or "
                         "5 (Zipf keys, 4 KB values, 256 partitions; any --gpus)")
    ap.add_argument("--c1-text-mb", type=int, default=100)
    ap.add_argument("--c3-segments", type=int, default=256)
    ap.add_argument("--c3-segment-mb", type=int, default=64)
    ap.add_argument("--c3-cpu-segments", type=int, default=16)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="config 2 on one GPU: write the last timed step's outputs to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    single = args.impl != "reference" and args.config not in (1, 3, 5) and args.gpus == 1 and world == 1
    if args.dump_outputs and not single:
        ap.error("--dump-outputs is implemented for the single-GPU config 2 run")
    if args.records is None:
        if args.config == 5:
            args.records = 4_000_000      # 16.4 GB of records per GPU
        else:
            args.records = 100_000_000 if (args.gpus == 1 and world == 1) else 125_000_000
    if args.warmup < 3 and args.impl != "reference":
        args.warmup = 3
    if args.impl == "reference":
        return reference_arm(args)
    if args.config == 1:
        return config1(args)
    if args.config == 3:
        return config3(args)
    if single:
        return single_gpu(args)
    if args.config == 5 and "RANK" not in os.environ:      # config 5 on one GPU without torchrun: a world of one
        os.environ.update({"RANK": "0", "WORLD_SIZE": "1", "LOCAL_RANK": "0", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29533"})
    from tez_b200 import multigpu_bench

    def verify_partition(runs, merged):
        # the checker (test infrastructure, outside the timed region): TezMerger restatement over the same runs
        import numpy as np
        from oracle import tez_oracle as O
        exp, _, _ = O.merge_ifile(runs, O.CMP_BYTES, factor=100)
        assert np.array_equal(np.frombuffer(merged, dtype=np.uint8), exp), "merged partition differs from the oracle's TezMerger output"

    return multigpu_bench.run(args, workload_config, ClockSampler, hbm_peak, run_cpu, host_cores, verify_partition)


if __name__ == "__main__":
    sys.exit(main())
