#!/usr/bin/env python
"""bench.py -- hot-path benchmark: prints one JSON result line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4]
                    [--rows R] [--dump-outputs DIR]

A "step" is one pass of convert_from_rows over the whole synthetic workload.
  value      : rows/s with the JCUDF row buffer already resident in HBM (CUDA events, max over ranks)
  e2e        : the same pass through the host-buffer C-ABI entry point (pinned host rows in, host
               columns out; H2D + kernel + D2H inside the timed region)
  roofline   : algorithmic bytes per launch / measured kernel time vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline: the oracle's threaded row->column loop (a stated stand-in for Spark's
               InternalRow->ColumnarBatch, BASELINE.md section 3) on a bounded sample, host cores
--impl reference times that CPU path alone (no JVM / libcudf in this image: the reference itself
cannot run, SURVEY.md 8c).
"""
from __future__ import annotations

import argparse
import ctypes
from ctypes import c_int32 as C_int32
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "spark-rapids-jni_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

# cudf type ids used by the workloads
INT8, INT16, INT32, INT64, FLOAT32, FLOAT64, BOOL8, TS_US, STRING, DEC32, DEC128 = 1, 2, 3, 4, 9, 10, 11, 15, 23, 25, 27
UINT8, UINT16, UINT64 = 5, 6, 8
SIZE = {INT8: 1, INT16: 2, INT32: 4, INT64: 8, FLOAT32: 4, FLOAT64: 8, BOOL8: 1, TS_US: 8, DEC32: 4, DEC128: 16,
        UINT8: 1, UINT16: 2, UINT64: 8}
# the reference's own nvbench shapes (src/main/cpp/benchmarks/row_conversion.cpp:27-147)
NVB_CYCLE = [INT8, INT32, INT16, INT64, INT32, BOOL8, UINT16, UINT8, UINT64]
NVB_CYCLE_STR = [INT8, INT32, INT16, INT64, INT32, BOOL8, STRING, UINT16, UINT8, UINT64]


def cycle(types, n):
    return [types[i % len(types)] for i in range(n)]

WORKLOADS = {
    # BASELINE.json configs[1]: 100M rows x 32 fixed-width cols convert_from_rows, 1xB200
    "c2": dict(name="C2: 100M rows x 32 fixed-width cols ([INT8,INT16,INT32,INT64,FLOAT32,FLOAT64,BOOL8,TIMESTAMP_US]x4) "
                    "convert_from_rows, 200 B rows, 20% nulls",
               types=[INT8, INT16, INT32, INT64, FLOAT32, FLOAT64, BOOL8, TS_US] * 4, rows=100_000_000, null_frac=0.2),
    # BASELINE.json configs[3]: store_sales, from_rows fused with xxhash64(ss_item_sk, ss_ticket_number)
    "c4": dict(name="C4: TPC-DS store_sales (23 cols, 104 B rows) convert_from_rows + xxhash64 partition key in one call",
               types=[INT32] * 9 + [INT64, INT32] + [DEC32] * 12, rows=400_000_000, null_frac=0.04, hash_keys=[1, 9]),
    # BASELINE.json configs[2]: 100M rows x 256 mixed cols (int32/int64/decimal128/utf8, 20% null), to+from rows.
    # ~390 GB of rows cannot be resident: a step streams 100M rows as `batches` x `batch_rows` conversions over a
    # resident pool of distinct <=2 GiB batches (each batch is what one LIST<INT8> column / one JNI call carries).
    # the reference's nvbench shapes, timed through the public API like nvbench's exec_tag::sync (allocation and the
    # size read-backs included): "Fixed Width Only" 212 columns, "Fixed or Variable Width" 155 columns +- STRING
    "nvbench_fixed": dict(name="nvbench 'Fixed Width Only': 212 cols cycling [INT8,INT32,INT16,INT64,INT32,BOOL8,UINT16,UINT8,UINT64] "
                               "(benchmarks/row_conversion.cpp:27-64)", types=cycle(NVB_CYCLE, 212), rows=1 << 20, null_frac=0.0, nvbench=True),
    "nvbench_nostr": dict(name="nvbench 'Fixed or Variable Width', no strings: 155 cols (benchmarks/row_conversion.cpp:66-147)",
                          types=cycle(NVB_CYCLE, 155), rows=1 << 20, null_frac=0.0, nvbench=True),
    "nvbench_var": dict(name="nvbench 'Fixed or Variable Width', include strings: 155 cols cycling [...,BOOL8,STRING,UINT16,...], "
                             "strings ~N(16,8) in [0,32] B (benchmarks/row_conversion.cpp:66-147)",
                        types=cycle(NVB_CYCLE_STR, 155), rows=1 << 20, null_frac=0.0, nvbench=True),
    # SURVEY 8f rank 1: the consumer of the row hashes -- Spark HashPartitioning of a device-resident store_sales batch
    "partition": dict(name="hash partition: TPC-DS store_sales (23 cols, 96 data B/row), pmod(murmur3_32(42, ss_item_sk, ss_ticket_number), 200) "
                           "+ stable partition of every column",
                      types=[INT32] * 9 + [INT64, INT32] + [DEC32] * 12, rows=100_000_000, null_frac=0.04, hash_keys=[1, 9], partitions=200,
                      partition=True),
    # the exchange step of the widened path: every GPU hash-partitions its store_sales batch, writes Kudo partitions, the
    # partitions travel with ONE all_to_all_single over NVLink (NCCL), every GPU assembles what it received
    "shuffle": dict(name="shuffle exchange: per GPU 50M store_sales rows (23 cols, 96 data B/row, 4% nulls) -> pmod(murmur3(ss_item_sk, "
                         "ss_ticket_number)) -> Kudo split -> all_to_all_single -> assemble; 8 partitions per GPU",
                    types=[INT32] * 9 + [INT64, INT32] + [DEC32] * 12, rows=50_000_000, null_frac=0.04, hash_keys=[1, 9], parts_per_rank=8,
                    shuffle=True),
    # SURVEY 8f rank 2: the Kudo shuffle wire format of the same store_sales batch, cut into 200 partitions
    "kudo": dict(name="Kudo split / assemble: TPC-DS store_sales (23 cols, 96 data B/row, 4% nulls), 200 partitions",
                 types=[INT32] * 9 + [INT64, INT32] + [DEC32] * 12, rows=100_000_000, null_frac=0.04, partitions=200, kudo=True),
    # SURVEY 8f rank 3: the same C2 table through Apache Spark's UnsafeRow format (264 B rows: 8 B bitset + 32 slots)
    "unsafe_c2": dict(name="UnsafeRow codec: 50M rows x 32 fixed-width cols ([INT8,INT16,INT32,INT64,FLOAT32,FLOAT64,BOOL8,TIMESTAMP_US]x4), "
                           "264 B UnsafeRows, 20% nulls", types=[INT8, INT16, INT32, INT64, FLOAT32, FLOAT64, BOOL8, TS_US] * 4,
                      rows=50_000_000, null_frac=0.2, unsafe=True),
    "c3": dict(name="C3: 100M rows x 256 mixed cols ([INT32,INT64,DECIMAL128,STRING]x64, 20% nulls, strings ~N(16,8) in [0,32] B) "
                    "convert_from_rows, streamed as 200 batches of 500K rows (<=2 GiB each)",
               types=[INT32, INT64, DEC128, STRING] * 64, rows=100_000_000, null_frac=0.2, batch_rows=500_000, pool=4),
}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def gpu_local_cpus(torch, index: int):
    """CPUs of the NUMA node the GPU hangs off (sysfs local_cpulist of its PCI function), or None."""
    try:
        pr = torch.cuda.get_device_properties(index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/local_cpulist") as f:
            txt = f.read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        return cpus or None
    except Exception:
        return None


class NumaBind:
    """Run the host side of the end-to-end leg on the GPU's NUMA node (what `numactl --cpunodebind` does for a
    Spark executor pinned to its GPU): pinned buffers are first-touched there and the PCIe copies do not cross
    the socket interconnect.  Restores the original affinity on exit (the CPU baseline uses every core)."""

    def __init__(self, torch, index: int):
        self.cpus = gpu_local_cpus(torch, index) if not os.environ.get("SRJ_BENCH_NO_NUMA") else None
        self.prev = None

    def __enter__(self):
        if self.cpus:
            try:
                self.prev = os.sched_getaffinity(0)
                os.sched_setaffinity(0, self.cpus & self.prev or self.prev)
            except Exception:
                self.prev = None
        return self

    def __exit__(self, *a):
        if self.prev:
            try:
                os.sched_setaffinity(0, self.prev)
            except Exception:
                pass
        return False


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def box_copy_gbs(torch):
    """STREAM-style copy on THIS box (same recipe as MEASURED_PEAKS.json: b.copy_(a), read+write bytes, best of 10).
    Reported for context only -- the roofline denominator stays the driver-measured peak."""
    a = torch.empty(1 << 30, dtype=torch.bfloat16, device="cuda")
    b = torch.empty_like(a)
    best = 0.0
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); b.copy_(a); e1.record()
        torch.cuda.synchronize()
        best = max(best, 2 * a.numel() * 2 / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del a, b
    return round(best, 1)


def algorithmic_bytes_per_row(types, row_size, hashed=False):
    """SURVEY 8(d): read the padded row + write every column element + ncols/8 mask bytes (+ 8 B hash)."""
    return row_size + sum(SIZE[t] for t in types) + len(types) / 8.0 + (8 if hashed else 0)


# ---------------------------------------------------------------------------------------------------
def synth_columns_gpu(torch, S, types, n, null_frac, seed):
    """Seeded synthetic columns on the device (data = random bytes; BOOL8 in {0,1}; masks ~null_frac nulls)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    cols = []
    words = (n + 31) // 32
    for t in types:
        sz = SIZE[t]
        data = torch.empty(n * sz, dtype=torch.uint8, device="cuda")
        step = 1 << 28
        for o in range(0, n * sz, step):          # chunked: randint materialises int64 internally
            m = min(step, n * sz - o)
            data[o:o + m] = torch.randint(0, 256, (m,), dtype=torch.uint8, device="cuda", generator=g)
        if t == BOOL8:
            data &= 1
        # valid with probability 1 - null_frac: compare a random byte per row, pack to words
        mask = torch.empty(words, dtype=torch.int32, device="cuda")
        wstep = 1 << 21
        weights = (1 << torch.arange(32, device="cuda", dtype=torch.int64))
        thr = int(round(null_frac * 256))
        for o in range(0, words, wstep):
            m = min(wstep, words - o)
            bits = (torch.randint(0, 256, (m, 32), dtype=torch.uint8, device="cuda", generator=g) >= thr)
            w = (bits.to(torch.int64) * weights).sum(dim=1)
            mask[o:o + m] = torch.where(w >= 2**31, w - 2**32, w).to(torch.int32)
        cols.append(S.ColumnVector(S.DType(t), n, data, mask))
    return cols


def build_rows_gpu(torch, S, N, plan, cols, n, row_size):
    """Produce the JCUDF rows of `cols` with OUR to_rows into ONE contiguous device buffer (the C ABI takes
    caller-owned batch buffers, so the <=2 GiB batches are laid back to back)."""
    import ctypes as C
    lib = N.lib()
    carr = (N.SrjColumn * len(cols))()
    for i, c in enumerate(cols):
        carr[i] = c._c()
    batches = (N.SrjRowBatch * 4096)()
    nb = C.c_int32(0)
    st = int(torch.cuda.current_stream().cuda_stream)
    N.check(lib.srj_to_rows_plan_batches(plan.handle, carr, n, None, batches, 4096, C.byref(nb), st))
    rows = torch.empty(n * row_size, dtype=torch.uint8, device="cuda")
    offs = torch.empty(n + nb.value, dtype=torch.int32, device="cuda")
    optrs, dptrs = (C.c_void_p * nb.value)(), (C.c_void_p * nb.value)()
    for b in range(nb.value):
        optrs[b] = offs.data_ptr() + 4 * (batches[b].row_start + b)
        dptrs[b] = rows.data_ptr() + batches[b].row_start * row_size
    N.check(lib.srj_convert_to_rows(plan.handle, carr, n, None, batches, nb.value, optrs, dptrs, st))
    torch.cuda.synchronize()
    return rows, nb.value


def run_ours(args, wl, rank, world):
    import ctypes as C

    import torch
    import torch.distributed as dist
    import srj_b200 as S
    from srj_b200 import _native as N

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    types = wl["types"]
    n = int(args.rows or wl["rows"])          # weak scaling: every rank converts the full per-GPU workload
    plan = S.Plan.get([S.DType(t) for t in types])
    row_size = plan.layout.fixed_row_size
    hashed = "hash_keys" in wl and os.environ.get("SRJ_BENCH_NOHASH") != "1"
    bpr = algorithmic_bytes_per_row(types, row_size, hashed)
    lib = N.lib()

    # ---- synthetic inputs (outside the timed region) ------------------------------------------------
    src = synth_columns_gpu(torch, S, types, n, wl["null_frac"], seed=42 + rank)
    rows, nbatches = build_rows_gpu(torch, S, N, plan, src, n, row_size)
    words = (n + 31) // 32
    outs = [S.ColumnVector(S.DType(t), n, torch.empty(n * SIZE[t], dtype=torch.uint8, device="cuda"),
                           torch.empty(words, dtype=torch.int32, device="cuda")) for t in types]
    carr = (N.SrjColumn * len(outs))()
    for i, c in enumerate(outs):
        carr[i] = c._c()
    nulls = torch.zeros(len(types), dtype=torch.int64, device="cuda")
    fh = None
    hout = None
    if hashed:
        fh = N.SrjFusedHash()
        fh.kind, fh.num_keys, fh.seed = N.HASH_XXHASH64, len(wl["hash_keys"]), 42
        for i, k in enumerate(wl["hash_keys"]):
            fh.key_columns[i] = k
        hout = torch.empty(n, dtype=torch.int64, device="cuda")
        fh.out = hout.data_ptr()
    stream = torch.cuda.current_stream()
    st = int(stream.cuda_stream)

    def step():
        N.check(lib.srj_convert_from_rows_fixed(plan.handle, rows.data_ptr(), None, rows.numel(), n, carr,
                                                nulls.data_ptr(), None, C.byref(fh) if fh else None, None, st))

    # correctness gate inside the bench: round trip equals the source columns (cheap, on device)
    step()
    torch.cuda.synchronize()
    for a, b in zip(outs, src):
        assert torch.equal(a.data, b.data) and torch.equal(a.mask, b.mask), "bench: from_rows(to_rows(x)) != x"
    del src

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    cuprof = os.environ.get("SRJ_CUPROF") == "1"      # ncu --profile-from-start off: capture the timed region only
    if cuprof:
        torch.cuda.cudart().cudaProfilerStart()
    t0.record(stream)
    for a, b in evs:
        a.record(stream)       # events on the launching stream: the conversion kernel is the only kernel between them
        step()
        b.record(stream)
    t1.record(stream)
    barrier()
    if cuprof:
        torch.cuda.cudart().cudaProfilerStop()
    clocks = sampler.stop() if rank == 0 else None
    total_ms = t0.elapsed_time(t1)
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    tt = torch.tensor([total_ms, kern_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms, kern_ms = float(tt[0]), float(tt[1])
    ms_per_step = total_ms / args.steps
    value = world * n / (ms_per_step * 1e-3)

    peak, peak_src = load_peaks()
    achieved = bpr * n / (kern_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": None,
                "kernel": "srj::from_rows_kernel" + (" + row_hash_stream_kernel over the key columns just written (one C-ABI call)" if wl.get("hash_keys") else ""),
                "kernel_ms": round(kern_ms, 4), "algorithmic_bytes_per_row": bpr, "rows_per_launch": n,
                "peak_source": peak_src, "this_box_copy_gbs": box_copy_gbs(torch) if rank == 0 else None}
    tr = os.path.join(ROOT, "profiles", f"traffic_{args.workload}.json")
    if os.path.exists(tr):
        try:
            j = json.load(open(tr))
            roofline["traffic"] = j["dram_bytes_per_launch"] * (n / j["rows_per_launch"])
            roofline["traffic_source"] = j.get("source")
        except Exception:
            pass

    # ---- multi-GPU config: NCCL all-gather of the per-column chunks over NVLink (north_star) ---------------
    # Each rank contributes the columns of its first n/world rows; every GPU ends with the n-row table.
    allgather = None
    if world > 1:
        from srj_b200 import sharding
        per = (n // world) // 32 * 32
        chunks = [c.data[: per * SIZE[t]] for c, t in zip(outs, types)] + [c.mask[: per // 32] for c in outs]
        gbytes = sum(ch.numel() * ch.element_size() for ch in chunks)
        fulls = sharding.gather_fixed_columns(dist, chunks, world)          # warm-up (allocates)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for ch, full in zip(chunks, fulls):
            dist.all_gather_into_tensor(full.view(-1), ch.contiguous().view(-1))
        g1.record(stream)
        barrier()
        tg = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        gms = float(tg[0])
        allgather = {"rows_per_rank": per, "bytes_sent_per_gpu": gbytes, "bytes_received_per_gpu": gbytes * (world - 1),
                     "ms": gms, "busbw_gbs": round(gbytes * (world - 1) / (gms * 1e-3) / 1e9, 1),
                     "collectives": len(chunks), "note": "one all_gather_into_tensor per column and per mask (NCCL)"}
        del fulls

    # ---- e2e: host rows -> host columns through the C-ABI host entry point --------------------------
    e2e = None
    cpu = None
    if not args.no_e2e:
        numa = NumaBind(torch, torch.cuda.current_device())
        with numa:
            h_rows = torch.empty(n * row_size, dtype=torch.uint8, pin_memory=True)
            h_rows.copy_(rows)
            torch.cuda.synchronize()
            h_cols = []
            harr = (N.SrjColumn * len(types))()
            for i, t in enumerate(types):
                d = torch.empty(n * SIZE[t], dtype=torch.uint8, pin_memory=True)
                m = torch.empty(words, dtype=torch.int32, pin_memory=True)
                h_cols.append((d, m))
                harr[i].type_id, harr[i].scale, harr[i].size = t, 0, n
                harr[i].data, harr[i].null_mask, harr[i].offsets = d.data_ptr(), m.data_ptr(), None
            h_nulls = np.zeros(len(types), np.int64)
            h2d = n * row_size
            d2h = sum(n * SIZE[t] + words * 4 for t in types) + 8 * len(types)

            def e2e_step():
                N.check(lib.srj_convert_from_rows_host(plan.handle, h_rows.data_ptr(), None, h_rows.numel(), n, harr,
                                                       h_nulls.ctypes.data, 0, None, None))

            e2e_step()                                   # warm-up (also validates)
            assert torch.equal(h_cols[3][0], outs[3].data.cpu()), "bench e2e: host result differs from device result"
            barrier()
            ksteps = max(1, min(args.steps, 3))
            w0 = time.perf_counter()
            for _ in range(ksteps):
                e2e_step()                               # synchronises internally (result is in host memory)
            barrier()
            e2e_s = (time.perf_counter() - w0) / ksteps
            te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            e2e = {"value": world * n / float(te[0]), "unit": "rows/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "steps": ksteps, "ms_per_step": float(te[0]) * 1e3, "api": "srj_convert_from_rows_host (pinned host buffers)",
                   "host_numa_bound": bool(numa.prev)}
        if rank == 0:
            cpu = cpu_baseline(types, row_size, h_rows.numpy(), min(n, args.cpu_sample_rows), bpr)
        del h_rows, h_cols

    if rank == 0:
        line = {"metric": "rows_per_sec_convert_from_rows", "value": value, "unit": "rows/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": wl["name"], "rows_per_gpu": n, "row_bytes": row_size, "columns": len(types),
                           "l2": "inputs+outputs (%.1f GB) >> 126 MB L2, no flush needed" % (bpr * n / 1e9),
                           "launch": "one srj_convert_from_rows_fixed call over all rows (C ABI takes int64 row counts; "
                                     "rows were produced by srj_convert_to_rows in %d <=2GiB batches)" % nbatches,
                           "sharding": "contiguous row range per GPU, no data-path collective"},
                "hbm_gbs": round(achieved, 1), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": args.steps * (2 if wl.get("hash_keys") else 1), "clocks": clocks}
        if allgather:
            line["allgather"] = allgather
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------
# C3: variable-width (strings + decimal128), streamed in <=2 GiB batches
# ---------------------------------------------------------------------------------------------------
def synth_strings_gpu(torch, S, n, null_frac, g):
    """STRING column: lengths ~ clamp(round(N(16, 8)), 0, 32), null strings have length 0, printable ASCII chars."""
    words = (n + 31) // 32
    valid = torch.rand(n, device="cuda", generator=g) >= null_frac
    lens = torch.clamp(torch.round(torch.randn(n, device="cuda", generator=g) * 8 + 16), 0, 32).to(torch.int64)
    lens = lens * valid
    offs = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    offs[1:] = torch.cumsum(lens, 0)
    total = int(offs[-1])
    chars = torch.randint(32, 127, (total,), dtype=torch.uint8, device="cuda", generator=g)
    pad = words * 32 - n
    bits = torch.cat([valid, torch.zeros(pad, dtype=torch.bool, device="cuda")]).view(words, 32).to(torch.int64)
    w = (bits * (1 << torch.arange(32, device="cuda", dtype=torch.int64))).sum(dim=1)
    mask = torch.where(w >= 2**31, w - 2**32, w).to(torch.int32)
    return S.ColumnVector(S.DType(STRING), n, chars, mask, offs.to(torch.int32))


def synth_c3_host(types, n, null_frac, seed):
    """One C3 batch on the HOST (numpy): same distributions as the device generator (fixed-width = random bytes,
    strings ~ clamp(round(N(16, 8)), 0, 32) printable ASCII, null strings have length 0)."""
    from oracle import oracle as O
    rng = np.random.Generator(np.random.Philox(seed))
    cols = []
    for t in types:
        valid = rng.random(n) >= null_frac
        mask = O.pack_mask(valid)
        if t == STRING:
            lens = np.clip(np.rint(rng.normal(16, 8, n)), 0, 32).astype(np.int64) * valid
            offs = np.zeros(n + 1, np.int32)
            np.cumsum(lens, out=offs[1:])
            cols.append(O.HCol(t, rng.integers(32, 127, int(offs[-1]), dtype=np.uint8), mask, offs, 0, n))
        else:
            cols.append(O.HCol(t, rng.integers(0, 256, n * SIZE[t], dtype=np.uint8), mask, None, -11 if t == DEC128 else 0, n))
    return cols


def gather_ranges(torch, buf, starts, lens):
    """buf[starts[0]:starts[0] + lens[0]] ++ buf[starts[1]:...] ++ ... (int64 device tensors), on the device."""
    ends = torch.cumsum(lens, 0)
    pos = torch.arange(int(ends[-1]), device=buf.device)
    pos += torch.repeat_interleave(starts - (ends - lens), lens)
    return buf[pos]


def dump_c3(dirname, torch, types, nb, outs, direction):
    """--dump-outputs: what the last timed step handed its caller, as DIR/<name>.npy (values exact in float64 / float32).
    A step cycles over the resident pool, so slot k holds the output of every round i with i % pool == k.  A slot is a
    whole batch of several GB: the same seeded sample of S rows of every slot is written.
      rows                              [S]            the sampled row indices of a batch
      from_rows: valid                  [pool, S, ncols]   validity bits
                 fixed_words            [pool, S, W]       the fixed-width values as little-endian int32 words, column order
                 string_starts, string_lengths [pool, S, nstr]  offsets[row] and offsets[row + 1] - offsets[row]
                 string_chars           [chars]            the chars of the sampled strings, slot, column, row order
      to_rows:   row_starts, row_lengths [pool, S]         offsets[row] and the row's length in bytes
                 row_words              [words]            the sampled rows as little-endian int32 words, slot, row order"""
    dev = outs[0]["cols"][0].mask.device if direction == "from_rows" else outs[0]["offs"].device
    rows = np.sort(np.random.default_rng(0).choice(nb, min(nb, 1024 if direction == "from_rows" else 512), replace=False))
    rows[0], rows[-1] = 0, nb - 1                          # the first and last row of a batch are always in the sample
    idx = torch.from_numpy(rows).to(dev)
    res = {"rows": rows.astype(np.float64)}
    if direction == "from_rows":
        valid, words, starts, lens, chars = [], [], [], [], []
        for o in outs:
            v, w, s_, l_ = [], [], [], []
            for c in o["cols"]:
                v.append((c.mask[idx // 32] >> (idx % 32).to(torch.int32)) & 1)
                if c.dtype.type_id == STRING:
                    offs = c.offsets.long()
                    s, n = offs[idx], offs[idx + 1] - offs[idx]
                    s_.append(s); l_.append(n)
                    chars.append(gather_ranges(torch, c.data, s, n))
                else:
                    w.append(c.data.view(nb, SIZE[c.dtype.type_id])[idx].contiguous().view(torch.int32))
            valid.append(torch.stack(v, 1))
            words.append(torch.cat(w, 1))
            starts.append(torch.stack(s_, 1))
            lens.append(torch.stack(l_, 1))
        res["valid"] = torch.stack(valid).cpu().numpy().astype(np.float32)
        res["fixed_words"] = torch.stack(words).cpu().numpy().astype(np.float64)
        res["string_starts"] = torch.stack(starts).cpu().numpy().astype(np.float64)
        res["string_lengths"] = torch.stack(lens).cpu().numpy().astype(np.float64)
        res["string_chars"] = torch.cat(chars).cpu().numpy().astype(np.float32)
    else:
        starts, lens, words = [], [], []
        for o in outs:
            offs = o["offs"].long()
            s, n = offs[idx], offs[idx + 1] - offs[idx]
            starts.append(s); lens.append(n)
            words.append(gather_ranges(torch, o["data"], s, n).view(torch.int32))   # JCUDF rows are 8-byte multiples
        res["row_starts"] = torch.stack(starts).cpu().numpy().astype(np.float64)
        res["row_lengths"] = torch.stack(lens).cpu().numpy().astype(np.float64)
        res["row_words"] = torch.cat(words).cpu().numpy().astype(np.float64)
    total = sum(a.nbytes for a in res.values())
    assert total <= 64 << 20, f"--dump-outputs: {total} bytes exceed 64 MB"
    os.makedirs(dirname, exist_ok=True)
    for name, a in res.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def run_c3(args, wl, rank, world):
    import ctypes as C

    import torch
    import torch.distributed as dist
    import srj_b200 as S
    from srj_b200 import _native as N

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    types = wl["types"]
    nc = len(types)
    nb = int(wl["batch_rows"])
    total_rows = int(args.rows or wl["rows"])
    # STRONG scaling (BASELINE configs[4]): the job is total_rows rows whatever N; a "round" converts one batch of nb
    # rows on every rank (the rank's contiguous row range of an N x nb-row global batch), then all-gathers the columns
    rounds = max(1, total_rows // (nb * world))
    pool = min(int(wl["pool"]), rounds)
    dts = [S.DType(t, -11 if t == DEC128 else 0) for t in types]
    plan = S.Plan.get(dts)
    lib = N.lib()
    stream = torch.cuda.current_stream()
    st = int(stream.cuda_stream)
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    words = (nb + 31) // 32
    do_gather = world > 1 and args.direction == "from_rows" and not args.no_gather

    # ---- resident pool of distinct batches: columns -> (our) to_rows -> rows ---------------------------
    batches = []
    for b in range(pool):
        cols = []
        fixed = synth_columns_gpu(torch, S, [t for t in types if t != STRING], nb, wl["null_frac"], seed=77 + 13 * b + 1000 * rank)
        fi = iter(fixed)
        for t in types:
            cols.append(synth_strings_gpu(torch, S, nb, wl["null_frac"], g) if t == STRING else next(fi))
        for c, d in zip(cols, dts):
            c.dtype = d
        rows = S.RowConversion.convertToRows(S.Table(cols))
        assert len(rows) == 1, "batch must fit one LIST column"
        batches.append(dict(cols=cols, rows=rows[0]))
    torch.cuda.synchronize()

    # algorithmic bytes of one from_rows batch (SURVEY 8d): rows as stored + 4 B row offsets, all column bytes out
    def alg_bytes(bt):
        rb = bt["rows"].child.size + 4 * (nb + 1)
        out = 0
        for c in bt["cols"]:
            out += words * 4
            out += (4 * (nb + 1) + c.data.numel()) if c.dtype.type_id == STRING else c.data.numel()
        return rb + out
    alg = [alg_bytes(bt) for bt in batches]
    alg_step = sum(alg[i % pool] for i in range(rounds))

    gather_info = None
    if args.direction == "from_rows":
        # Outputs of a slot live in ONE packed slab: [fixed-width data | STRING offsets] per column, the masks, the
        # phase-1 totals (nc + 1 int64) and the chars of the STRING columns back to back -- what the rank contributes to
        # the all-gather is one contiguous buffer, so the collective is ONE ncclAllGather per round.
        from srj_b200 import sharding
        chars_need = [sum((c.data.numel() + 15) & ~15 for c in bt["cols"] if c.dtype.type_id == STRING) for bt in batches]
        cap = torch.tensor([max(chars_need)], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(cap, op=dist.ReduceOp.MAX)          # common chars capacity (equal counts for the all-gather)
        lay = sharding.SlabLayout([0 if t == STRING else SIZE[t] for t in types], nb, int(cap[0]))
        at_data, at_mask, at_tot, at_chars, slab_bytes = lay.at_data, lay.at_mask, lay.at_totals, lay.at_chars, lay.nbytes
        outs = []
        for bt in batches:
            slab = torch.empty(slab_bytes, dtype=torch.uint8, device="cuda")
            o, co = [], at_chars
            for i, c in enumerate(bt["cols"]):
                m = slab[at_mask[i]: at_mask[i] + words * 4].view(torch.int32)
                if c.dtype.type_id == STRING:
                    offs = slab[at_data[i]: at_data[i] + (nb + 1) * 4].view(torch.int32)
                    o.append(S.ColumnVector(c.dtype, nb, slab[co: co + c.data.numel()], m, offs))
                    co += (c.data.numel() + 15) & ~15
                else:
                    o.append(S.ColumnVector(c.dtype, nb, slab[at_data[i]: at_data[i] + c.data.numel()], m))
            carr = (N.SrjColumn * len(o))()
            for i, c in enumerate(o):
                carr[i] = c._c()
            outs.append(dict(cols=o, carr=carr, slab=slab, totals=slab[at_tot: at_tot + (nc + 1) * 8].view(torch.int64)))
        nulls = torch.zeros(nc, dtype=torch.int64, device="cuda")
        wsb = lib.srj_from_rows_workspace_bytes(plan.handle, nb)
        wss = [torch.empty(max(wsb, 8), dtype=torch.uint8, device="cuda") for _ in range(pool)]   # one workspace per call pair

        def convert(i):
            k = i % pool
            rv, o = batches[k]["rows"], outs[k]
            N.check(lib.srj_convert_from_rows_fixed(plan.handle, rv.child.data.data_ptr(), rv.offsets.data_ptr(), rv.child.size,
                                                    nb, o["carr"], nulls.data_ptr(), o["totals"].data_ptr(), None, wss[k].data_ptr(), st))
            N.check(lib.srj_convert_from_rows_strings(plan.handle, rv.child.data.data_ptr(), rv.offsets.data_ptr(), rv.child.size,
                                                      nb, o["carr"], o["totals"].data_ptr(), wss[k].data_ptr(), st))
        kernels_per_batch = 3        # from_rows_wide_kernel, wide_group_scan_kernel, strings_wide_kernel
        metric = "rows_per_sec_convert_from_rows"
    else:
        # to_rows: plan (row sizes + scan; its size read-back is part of the API) + convert into preallocated buffers
        outs = []
        for bt in batches:
            rv = bt["rows"]
            carr = (N.SrjColumn * len(types))()
            for i, c in enumerate(bt["cols"]):
                carr[i] = c._c()
            ws = torch.empty(max(8, lib.srj_to_rows_workspace_bytes(plan.handle, nb)), dtype=torch.uint8, device="cuda")
            outs.append(dict(carr=carr, ws=ws, offs=torch.empty(nb + 1, dtype=torch.int32, device="cuda"),
                             data=torch.empty(rv.child.size, dtype=torch.uint8, device="cuda")))
        rb = (N.SrjRowBatch * 8)()
        nbo = C.c_int32(0)

        def convert(i):
            o = outs[i % pool]
            N.check(lib.srj_to_rows_plan_batches(plan.handle, o["carr"], nb, o["ws"].data_ptr(), rb, 8, C.byref(nbo), st))
            op, dp = (C.c_void_p * 1)(o["offs"].data_ptr()), (C.c_void_p * 1)(o["data"].data_ptr())
            N.check(lib.srj_convert_to_rows(plan.handle, o["carr"], nb, o["ws"].data_ptr(), rb, 1, op, dp, st))
        kernels_per_batch = 4 + 1
        metric = "rows_per_sec_convert_to_rows"

    # correctness gate: every pool batch round-trips
    for i in range(pool):
        convert(i)
    torch.cuda.synchronize()
    for i in range(pool):
        if args.direction == "from_rows":
            for a, b in zip(outs[i]["cols"], batches[i]["cols"]):
                assert torch.equal(a.mask, b.mask), "bench c3: mask mismatch"
                if a.dtype.type_id == STRING:
                    assert torch.equal(a.offsets, b.offsets) and torch.equal(a.data, b.data), "bench c3: string mismatch"
                else:
                    assert torch.equal(a.data, b.data), "bench c3: data mismatch"
        else:
            assert torch.equal(outs[i]["data"], batches[i]["rows"].child.data), "bench c3: row bytes mismatch"
            assert torch.equal(outs[i]["offs"], batches[i]["rows"].offsets), "bench c3: row offsets mismatch"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- multi-GPU: one all-gather of the packed slab per round, overlapped with the next round's conversion -------
    if do_gather:
        peer = None
        if args.gather == "p2p":
            try:
                peer = sharding.PeerGather(dist, slab_bytes, world, rank, torch.device("cuda", local))
                gbuf = peer.bufs
            except Exception as ex:                   # symmetric memory unavailable: fall back to the NCCL collective
                if rank == 0:
                    print("bench: peer-memory gather unavailable (%s); using ncclAllGather" % ex, file=sys.stderr)
                peer = None
        if peer is None:
            gbuf = [torch.empty(world * slab_bytes, dtype=torch.uint8, device="cuda") for _ in range(2)]
        pre, post = torch.cuda.Stream(), torch.cuda.Stream()
        ev_conv = [torch.cuda.Event() for _ in range(pool)]
        ev_done = [None] * pool                      # gather + rebase of the slot's last use finished
        ev_gfree = [None, None]                      # the gathered buffer has been consumed (rebase done)
        sidx = [i for i, t in enumerate(types) if t == STRING]
        d_offs_at = torch.tensor([at_data[i] for i in sidx], dtype=torch.int64, device="cuda")
        d_scol = torch.tensor(sidx, dtype=torch.int32, device="cuda")

        def gather(i):
            k, gb = i % pool, i % 2
            ev_conv[k].record(stream)
            if peer is not None:
                if ev_gfree[gb] is not None:
                    peer.main.wait_event(ev_gfree[gb])
                landed = peer.gather(outs[k]["slab"], gb, ev_conv[k])     # copy engines over NVLink peer memory
                post.wait_event(landed)
            else:
                pre.wait_event(ev_conv[k])
                if ev_gfree[gb] is not None:
                    pre.wait_event(ev_gfree[gb])
                with torch.cuda.stream(pre):
                    _, work = sharding.gather_slab(dist, outs[k]["slab"], world, out=gbuf[gb], async_op=True)   # ONE ncclAllGather
            with torch.cuda.stream(post):
                if peer is None:
                    work.wait()
                gt = gbuf[gb].view(world, slab_bytes)[:, at_tot: at_tot + (nc + 1) * 8].contiguous().view(torch.int64)
                N.check(lib.srj_shard_rebase_offsets(gbuf[gb].data_ptr(), slab_bytes, d_offs_at.data_ptr(), d_scol.data_ptr(),
                                                     gt.data_ptr(), nb, nc, len(sidx), world, int(post.cuda_stream)))
                e = torch.cuda.Event()
                e.record(post)
            ev_done[k], ev_gfree[gb] = e, e

        # check the gathered table once: rank r's chunk of every column equals what rank r converted
        convert(0)
        gather(0)
        torch.cuda.synchronize()
        mine = gbuf[0].view(world, slab_bytes)[rank]
        i0 = next(i for i, t in enumerate(types) if t != STRING)
        assert torch.equal(mine[at_data[i0]: at_data[i0] + nb * SIZE[types[i0]]], outs[0]["cols"][i0].data), "bench c5: gathered chunk differs"
        barrier()

    def step(with_gather):
        for i in range(rounds):
            k = i % pool
            if with_gather and ev_done[k] is not None:
                stream.wait_event(ev_done[k])        # the slot's slab is free again
            convert(i)
            if with_gather:
                gather(i)
        if with_gather:
            stream.wait_stream(post)

    def timed(with_gather, steps):
        for _ in range(args.warmup):
            step(with_gather)
        barrier()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for _ in range(steps):
            step(with_gather)
        t1.record(stream)
        barrier()
        tt = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt[0]) / steps

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    cuprof = os.environ.get("SRJ_CUPROF") == "1"
    if cuprof:
        torch.cuda.cudart().cudaProfilerStart()
    ms_convert = timed(False, args.steps)                         # conversion only (no collective)
    if cuprof:
        torch.cuda.cudart().cudaProfilerStop()
    ms_gather = timed(True, args.steps) if do_gather else None    # conversion + all-gather, inside the step
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_c3(args.dump_outputs, torch, types, nb, outs, args.direction)
    ms_per_step = ms_gather if do_gather else ms_convert
    rows_step = rounds * nb                                       # rows one rank converts per step
    value = world * rows_step / (ms_per_step * 1e-3)
    peak, peak_src = load_peaks()
    achieved = alg_step / (ms_convert * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": None, "kernel": "whole conversion of a batch: from_rows_wide_kernel + wide_group_scan_kernel + strings_wide_kernel"
                if args.direction == "from_rows" else "whole conversion of a batch (all kernels of the two C-ABI calls)",
                "algorithmic_bytes_per_row": alg_step / rows_step, "rows_per_launch": nb, "peak_source": peak_src,
                "ms_per_batch": ms_convert / rounds, "per_gpu": True}
    tr = os.path.join(ROOT, "profiles", "traffic_c3.json")
    if os.path.exists(tr) and args.direction == "from_rows":
        try:
            j = json.load(open(tr))
            roofline["traffic"] = j["dram_bytes_per_launch"] * (nb / j["rows_per_launch"])
            roofline["traffic_source"] = j.get("source")
        except Exception:
            pass
    if do_gather:
        sent = slab_bytes
        gms = max(ms_gather - ms_convert, 1e-9) / rounds
        gather_info = {"collective": ("all-gather of the rank's packed slab per round over NVLink peer memory (symmetric memory, "
                                      "copy engines: no SM taken from the conversion kernels)" if peer is not None else
                                      "one ncclAllGather of the rank's packed slab per round") +
                                     " (columns + masks + STRING offsets + totals + chars), overlapped with the next round's "
                                     "conversion; STRING offsets rebased by srj_shard_rebase_offsets",
                       "transport": "p2p-copy-engine" if peer is not None else "nccl",
                       "bytes_sent_per_gpu_per_round": sent, "bytes_received_per_gpu_per_round": sent * (world - 1),
                       "rounds_per_step": rounds, "ms_per_step_convert_only": ms_convert, "ms_per_step_convert_plus_gather": ms_gather,
                       "rows_per_sec_convert_only": world * rows_step / (ms_convert * 1e-3),
                       "rows_per_sec_convert_plus_gather": world * rows_step / (ms_gather * 1e-3),
                       "busbw_gbs": round(sent * (world - 1) / ((ms_gather / rounds) * 1e-3) / 1e9, 1),
                       "exposed_gather_ms_per_round": gms}

    phases = None
    if args.direction == "from_rows" and os.environ.get("SRJ_BENCH_PHASES") == "1":
        # diagnostics: the two C-ABI calls of a batch timed separately (events around each call, 3 passes over the pool)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        acc = [0.0, 0.0]
        cnt = 0
        for i in range(3 * pool):
            k = i % pool
            rv, o = batches[k]["rows"], outs[k]
            ev[0].record(stream)
            N.check(lib.srj_convert_from_rows_fixed(plan.handle, rv.child.data.data_ptr(), rv.offsets.data_ptr(), rv.child.size,
                                                    nb, o["carr"], nulls.data_ptr(), o["totals"].data_ptr(), None, wss[k].data_ptr(), st))
            ev[1].record(stream)
            N.check(lib.srj_convert_from_rows_strings(plan.handle, rv.child.data.data_ptr(), rv.offsets.data_ptr(), rv.child.size,
                                                      nb, o["carr"], o["totals"].data_ptr(), wss[k].data_ptr(), st))
            ev[2].record(stream)
            torch.cuda.synchronize()
            acc[0] += ev[0].elapsed_time(ev[1]); acc[1] += ev[1].elapsed_time(ev[2]); cnt += 1
        phases = {"phase1_ms": acc[0] / cnt, "phase2_ms": acc[1] / cnt}

    # ---- e2e through the public API with HOST buffers: pinned host rows -> device -> RowConversion.convertFromRows
    # (incl. its size read-back) -> pinned host columns; a bounded number of batches, same batches as above ------
    e2e = None
    cpu = None
    if not args.no_e2e and args.direction == "from_rows":
        e2e = e2e_c3(args, torch, dist, S, batches, dts, nb, words, pool, rank, world, barrier)
        if rank == 0 and world == 1:
            cpu = cpu_baseline_c3(batches[0], types, nb, words)

    if rank == 0:
        line = {"metric": metric, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": wl["name"] + ("; row-range sharded over %d GPUs with one NCCL all-gather of the column "
                                                     "chunks per round (BASELINE configs[4])" % world if do_gather else ""),
                           "direction": args.direction, "total_rows_per_step": world * rows_step,
                           "rows_per_step_per_gpu": rows_step, "batch_rows": nb, "rounds_per_step": rounds,
                           "resident_pool_batches": pool, "avg_row_bytes": batches[0]["rows"].child.size / nb,
                           "sharding": "contiguous row range per GPU" + (", all-gather inside the timed step" if do_gather else
                                                                         ", no collective (single GPU or --no-gather)"),
                           "l2": "each batch touches ~%.1f GB >> 126 MB L2; pool of %d distinct batches" % (alg[0] / 1e9, pool)},
                "hbm_gbs": round(achieved, 1), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": args.steps * rounds * kernels_per_batch, "clocks": clocks}
        if gather_info:
            line["allgather"] = gather_info
        if phases:
            line["phases"] = phases
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def e2e_c3(args, torch, dist, S, batches, dts, nb, words, pool, rank, world, barrier):
    """Host rows -> host columns through the C ABI's host-buffer entry point (srj_convert_from_rows_host: pinned host
    rows in, pinned host columns out; the H2D of the rows, both conversion phases incl. the size read-back and the D2H of
    every output buffer happen inside the call), two batches in flight on two host threads the way concurrent Spark
    tasks share a GPU (the H2D of one batch overlaps the D2H of the other: PCIe is full duplex)."""
    from srj_b200 import hostpath
    kb = min(pool, 4)
    h_in, h_out = [], []
    for i in range(kb):
        rv = batches[i]["rows"]
        h_in.append((rv.child.data.cpu().pin_memory(), rv.offsets.cpu().pin_memory()))
        h_out.append(None)
    dev = torch.cuda.current_device()

    def e2e_batch(i):
        with torch.cuda.device(dev):
            a, b = h_in[i]
            h_out[i] = hostpath.convert_from_rows_host(a, b, nb, dts, out=h_out[i])      # one C call; buffers reused
    for i in range(kb):
        e2e_batch(i)                                                                       # warm-up: allocates the buffers
    c0 = batches[0]["cols"]
    assert torch.equal(h_out[0].data[3], c0[3].data.cpu()) and torch.equal(h_out[0].offsets[3], c0[3].offsets.cpu()), "bench e2e: host result differs"
    assert torch.equal(h_out[0].data[2], c0[2].data.cpu()), "bench e2e: host result differs"
    h2d = sum(a.numel() + 4 * b.numel() for a, b in h_in)
    d2h = sum(sum(d.numel() for d in o.data) + sum(4 * m.numel() for m in o.mask) + sum(4 * x.numel() for x in o.offsets if x is not None)
              for o in h_out)
    barrier()
    reps = 2

    def worker(w):
        for r in range(reps):
            for i in range(w, kb, 2):
                e2e_batch(i)
    w0 = time.perf_counter()
    th = [threading.Thread(target=worker, args=(w,)) for w in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    torch.cuda.synchronize()
    barrier()
    e2e_s = time.perf_counter() - w0
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    return {"value": world * reps * kb * nb / float(te[0]), "unit": "rows/s", "h2d_bytes_per_step": h2d * reps,
            "d2h_bytes_per_step": d2h * reps, "steps": 1, "ms_per_step": float(te[0]) * 1e3,
            "api": "srj_convert_from_rows_host (C ABI, pinned host rows in / pinned host columns out) on %d batches of %d rows "
                   "x %d passes, 2 host threads (2 batches in flight)" % (kb, nb, reps)}


def cpu_baseline_c3(batch, types, nb, words, nthreads=None):
    """The oracle's threaded from_rows over one batch of the same workload (rank 0, N=1)."""
    from oracle import oracle as O
    rv = batch["rows"]
    rvh, offh = rv.child.data.cpu().numpy(), rv.offsets.cpu().numpy()
    nthreads = nthreads or os.cpu_count()
    hc = [O.HCol(t, np.empty(max(c.data.numel(), 1), np.uint8), np.empty(words, np.uint32),
                 np.empty(nb + 1, np.int32) if t == STRING else None, 0, nb) for t, c in zip(types, batch["cols"])]
    O.from_rows_mt(rvh, offh, nb, hc, nthreads)
    times = []
    while sum(times) < 10.0 and len(times) < 20:
        t0_ = time.perf_counter()
        O.from_rows_mt(rvh, offh, nb, hc, nthreads)
        times.append(time.perf_counter() - t0_)
    best = min(times)
    return {"value": nb / best, "unit": "rows/s", "cores": nthreads, "kind": "port",
            "sample": "one %d-row batch of the same workload, best of %d passes (mean %.1f ms), %d OpenMP threads "
                      "(oracle/srj_oracle.c orc_from_rows_mt: fixed fields + lengths, per-column scan, chars)"
                      % (nb, len(times), 1e3 * sum(times) / len(times), nthreads),
            "ms_per_pass": best * 1e3}


def run_nvbench(args, wl, rank, world):
    """The reference's nvbench shapes through the PUBLIC API (RowConversion.convertToRows / convertFromRows: output
    allocation, batch planning and size read-backs inside the timed call, as nvbench's exec_tag::sync measures them)."""
    import torch
    import srj_b200 as S
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
    types = wl["types"]
    n = int(args.rows or wl["rows"])
    g = torch.Generator(device="cuda").manual_seed(5)
    fixed = iter(synth_columns_gpu(torch, S, [t for t in types if t != STRING], n, wl["null_frac"], seed=11))
    cols = [synth_strings_gpu(torch, S, n, wl["null_frac"], g) if t == STRING else next(fixed) for t in types]
    dts = [c.dtype for c in cols]
    tbl = S.Table(cols)
    rows = S.RowConversion.convertToRows(tbl)
    r0 = 0
    for rb in rows:                                   # > 2 GiB of rows come back as several LIST columns
        back = S.RowConversion.convertFromRows(rb, dts)
        for a, c in zip(back.columns, cols):
            if c.offsets is None:
                sz = c.dtype.size_in_bytes()
                assert torch.equal(a.data, c.data[r0 * sz:(r0 + rb.size) * sz]), "nvbench shape: round trip differs"
        r0 += rb.size
    row_bytes = sum(r.child.size for r in rows)
    col_bytes = sum(c.data.numel() + ((n + 31) // 32) * 4 + (4 * (n + 1) if c.offsets is not None else 0) for c in cols)
    alg = row_bytes + 4 * (n + 1) * (STRING in types) + col_bytes
    res = {}
    for direction in ("to_rows", "from_rows"):
        fn = (lambda: S.RowConversion.convertToRows(tbl)) if direction == "to_rows" else \
             (lambda: [S.RowConversion.convertFromRows(r, dts) for r in rows])
        for _ in range(max(3, args.warmup)):
            fn()
        torch.cuda.synchronize()
        times = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        res[direction] = float(np.median(times))
    peak, peak_src = load_peaks()
    sec = res[args.direction]
    print(json.dumps({"metric": "rows_per_sec_convert_" + args.direction, "value": n / sec, "unit": "rows/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": sec * 1e3, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                      "config": {"workload": wl["name"], "rows": n, "columns": len(types), "direction": args.direction,
                                 "timing": "host wall clock around the public API call + synchronize (allocation and read-backs included)"},
                      "roofline": {"bound": "hbm", "achieved": round(alg / sec / 1e9, 1), "peak": peak, "unit": "GB/s",
                                   "frac": round(alg / sec / 1e9 / peak, 4), "traffic": None, "kernel": "whole public-API call",
                                   "peak_source": peak_src},
                      "both_directions_ms": {k: v * 1e3 for k, v in res.items()}, "cpu_baseline": None, "e2e": None,
                      "gpu_launches": args.steps, "clocks": None}))


def cpu_baseline(types, row_size, h_rows_np, sample_rows, bpr, steps=None, nthreads=None):
    """Oracle's threaded row->column loop on a bounded sample of the same rows (host cores)."""
    from oracle import oracle as O
    nthreads = nthreads or os.cpu_count()
    n = int(sample_rows)
    cols = [O.HCol(t, np.empty(n * SIZE[t], np.uint8), np.empty((n + 31) // 32, np.uint32), None, 0, n) for t in types]
    data = h_rows_np[: n * row_size]
    O.from_rows_fixed_mt(data, n, cols, nthreads)            # warm-up / page-in
    reps, t_total = 0, 0.0
    while (t_total < 10.0 and reps < 50) if steps is None else reps < steps:
        t0 = time.perf_counter()
        O.from_rows_fixed_mt(data, n, cols, nthreads)
        t_total += time.perf_counter() - t0
        reps += 1
    sec = t_total / reps
    return {"value": n / sec, "unit": "rows/s", "cores": nthreads, "kind": "port",
            "sample": f"{n} rows of the same workload x {reps} passes, {nthreads} OpenMP threads over row ranges "
                      f"(oracle/srj_oracle.c orc_from_rows_fixed_mt), {bpr * n / sec / 1e9:.1f} GB/s algorithmic",
            "ms_per_pass": sec * 1e3}


def synth_columns_host(types, n, null_frac, seed):
    """The host twin of synth_columns_gpu for the CPU baselines of the 8(f) workloads (fixed-width columns)."""
    from oracle import oracle as O
    rng = np.random.default_rng(seed)
    cols = []
    for t in types:
        data = rng.integers(0, 256, n * SIZE[t], dtype=np.uint8)
        if t == BOOL8:
            data &= 1
        cols.append(O.HCol(t, data, O.pack_mask(rng.random(n) >= null_frac), None, 0, n))
    return cols


def cpu_baseline_f(kind, types, null_frac, n, hash_keys=None, P=200):
    """Single-core numpy / C-oracle port of one 8(f) step on a bounded sample of the same workload (rank 0, N = 1):
    kind = partition (murmur3 ids + stable argsort + take of every column), kudo_split, kudo_assemble,
    unsafe_to / unsafe_from (fixed-width rows)."""
    from oracle import kudo as K
    from oracle import oracle as O
    from oracle import unsafe_row as U
    cols = synth_columns_host(types, n, null_frac, 42)
    splits = np.linspace(0, n, P + 1).astype(np.int64)
    if kind == "kudo_assemble":
        buf, offs = K.split(cols, splits)
    if kind == "unsafe_from":
        rows = U.to_unsafe_rows_fixed(cols)
        bs = U.bitset_bytes(len(types))

    def once():
        if kind == "partition":
            ids = O.partition_ids([cols[i] for i in hash_keys], P, 42)
            return O.stable_partition(cols, ids, P)
        if kind == "kudo_split":
            return K.split(cols, splits)
        if kind == "kudo_assemble":
            return K.assemble(buf, offs, types)
        if kind == "unsafe_to":
            return U.to_unsafe_rows_fixed(cols)
        out = []                                        # unsafe_from: slots -> columns + masks
        for f, t in enumerate(types):
            out.append(np.ascontiguousarray(rows[:, bs + 8 * f: bs + 8 * f + SIZE[t]]))
            out.append(np.packbits(((rows[:, f // 64 * 8 + (f % 64) // 8] >> (f % 8)) & 1) ^ 1, bitorder="little"))
        return out

    once()
    times = []
    while sum(times) < 8.0 and len(times) < 10:
        t0 = time.perf_counter()
        once()
        times.append(time.perf_counter() - t0)
    best = min(times)
    return {"value": n / best, "unit": "rows/s", "cores": 1, "kind": "port",
            "sample": f"{n} rows of the same workload, best of {len(times)} passes, one core: numpy restatement of the step "
                      f"(oracle/oracle.py, oracle/kudo.py, oracle/unsafe_row.py; murmur3 in oracle/srj_oracle.c)",
            "ms_per_pass": best * 1e3}


def _cpu_f(kind, wl, n, **kw):
    try:
        return cpu_baseline_f(kind, wl["types"], wl["null_frac"], n, **kw)
    except Exception as e:                               # the baseline must never take the bench line down
        return {"value": None, "unit": "rows/s", "cores": 1, "kind": "port", "sample": f"failed: {e!r}"}


def run_partition(args, wl, rank, world):
    """Spark HashPartitioning step on one GPU: ids + stable partition maps + moving every column, inputs resident in HBM."""
    import ctypes as C
    import torch
    sys.path.insert(0, os.path.join(ROOT, "spark-rapids-jni_b200"))
    import srj_b200 as S
    from srj_b200 import _native as N
    torch.cuda.set_device(0)
    types, n, P = wl["types"], args.rows or wl["rows"], wl["partitions"]
    cols = synth_columns_gpu(torch, S, types, n, wl["null_frac"], 42)
    keys = [cols[i] for i in wl["hash_keys"]]
    words = (n + 31) // 32
    outs = [S.ColumnVector(c.dtype, n, torch.empty_like(c.data), torch.empty(words, dtype=torch.int32, device="cuda")) for c in cols]
    lib = N.lib()
    ws = torch.empty(lib.srj_partition_workspace_bytes(n, P), dtype=torch.uint8, device="cuda")
    ids = torch.empty(n, dtype=torch.int32, device="cuda")
    offs = torch.empty(P + 1, dtype=torch.int32, device="cuda")
    smap = torch.empty(n, dtype=torch.int32, device="cuda")
    gmap = torch.empty(n, dtype=torch.int32, device="cuda")
    nulls = torch.zeros(len(cols), dtype=torch.int64, device="cuda")
    karr = (N.SrjColumn * len(keys))(*[k._c() for k in keys])
    cin = (N.SrjColumn * len(cols))(*[c._c() for c in cols])
    cout = (N.SrjColumn * len(cols))(*[c._c() for c in outs])
    stream = torch.cuda.current_stream()
    st = int(stream.cuda_stream)

    def plan_step():
        N.check(lib.srj_hash_partition(karr, len(keys), n, C.c_uint32(42), P, ids.data_ptr(), offs.data_ptr(), smap.data_ptr(), gmap.data_ptr(),
                                       ws.data_ptr(), st))

    def step():
        plan_step()
        N.check(lib.srj_partition_columns(cin, cout, len(cols), n, P, smap.data_ptr(), gmap.data_ptr(), nulls.data_ptr(), ws.data_ptr(), st))

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    # size-independent check: the output is the input permuted by the gather map, partition by partition
    k0 = cols[9].data.view(torch.int64)
    assert torch.equal(outs[9].data.view(torch.int64), k0[gmap.long()]) and int(offs[P]) == n
    sampler = ClockSampler(0)
    sampler.start()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    e[0].record(stream)
    for _ in range(args.steps):
        plan_step()
    e[1].record(stream)
    for _ in range(args.steps):
        step()
    e[2].record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    plan_ms = e[0].elapsed_time(e[1]) / args.steps
    ms = e[1].elapsed_time(e[2]) / args.steps
    peak, peak_src = load_peaks()
    data_b = sum(SIZE[t] for t in types)
    bpr = 2 * (data_b + len(types) / 8.0) + 4          # read the table + write it partitioned + the ids
    gbs = bpr * n / (ms * 1e-3) / 1e9
    print(json.dumps({"metric": "rows_per_sec_hash_partition", "value": n / (ms * 1e-3), "unit": "rows/s", "n_gpus": 1, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "u8", "data": "synthetic",
                      "config": {"workload": wl["name"], "rows": n, "partitions": P, "l2": "inputs 9.6 GB >> 126 MB L2"},
                      "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": peak, "unit": "GB/s", "frac": round(gbs / peak, 4),
                                   "traffic": None, "kernel": "whole step: murmur3 + ids/histogram + scan + ranks + 23 column scatters + 23 mask gathers",
                                   "algorithmic_bytes_per_row": bpr, "peak_source": peak_src, "plan_only_ms": plan_ms},
                      "cpu_baseline": _cpu_f("partition", wl, 4_000_000, hash_keys=wl["hash_keys"], P=P), "e2e": None, "gpu_launches": args.steps * (6 + 2 * len(types)), "clocks": clocks}))


def run_shuffle(args, wl, rank, world):
    """The multi-GPU exchange of the widened path through its public API (srj_b200.shuffle.ShuffleExchange), device-resident
    input, weak scaling (rows per GPU fixed).  The collective (all_to_all_single) is inside the timed step."""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(ROOT, "spark-rapids-jni_b200"))
    import srj_b200 as S
    from srj_b200.shuffle import ShuffleExchange
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29517")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    types, n, k = wl["types"], args.rows or wl["rows"], wl["parts_per_rank"]
    cols = synth_columns_gpu(torch, S, types, n, wl["null_frac"], 42 + rank)
    table = S.Table(cols)
    ex = ShuffleExchange()
    stream = torch.cuda.current_stream()

    def step():
        return ex.shuffle(table, wl["hash_keys"], parts_per_rank=k)

    out = step()
    tot = torch.tensor([out.getRowCount()], dtype=torch.int64, device="cuda")
    dist.all_reduce(tot)
    assert int(tot[0]) == n * world, "rows were lost or duplicated in the exchange"
    del out
    for _ in range(args.warmup):
        step()
    dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    if rank == 0:
        peak, peak_src = load_peaks()
        data_b = sum(SIZE[t_] for t_ in types) + len(types) / 8.0
        # table read + partitioned copy written and read + buffer written; buffer read + assembled table written on the other side
        bpr = 6 * data_b
        gbs = bpr * n / (ms * 1e-3) / 1e9
        sent = data_b * n * (world - 1) / world                     # bytes a rank sends over NVLink per step
        print(json.dumps({"metric": "rows_per_sec_shuffle_exchange", "value": n * world / (ms * 1e-3), "unit": "rows/s", "n_gpus": world,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                          "config": {"workload": wl["name"], "rows_per_gpu": n, "partitions": world * k,
                                     "collective": "torch.distributed.all_to_all_single (NCCL) inside the timed step",
                                     "l2": "every pass touches >= 4.8 GB per GPU >> 126 MB L2"},
                          "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": peak, "unit": "GB/s", "frac": round(gbs / peak, 4),
                                       "traffic": None, "kernel": "whole step per GPU: murmur3 + partition plan + column moves + kudo split + all-to-all + assemble",
                                       "algorithmic_bytes_per_row": bpr, "peak_source": peak_src, "per_gpu": True,
                                       "nvlink_send_gbs_per_gpu": round(sent / (ms * 1e-3) / 1e9, 1)},
                          "cpu_baseline": None, "e2e": None, "gpu_launches": args.steps * 70, "clocks": clocks}))
    dist.destroy_process_group()


def run_kudo(args, wl, rank, world):
    """shuffle_split / shuffle_assemble of a device-resident table; --direction to_rows = split (default), from_rows = assemble."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "spark-rapids-jni_b200"))
    import srj_b200 as S
    from srj_b200 import _native as N
    torch.cuda.set_device(0)
    types, n, P = wl["types"], args.rows or wl["rows"], wl["partitions"]
    cols = synth_columns_gpu(torch, S, types, n, wl["null_frac"], 42)
    lib = N.lib()
    st = int(torch.cuda.current_stream().cuda_stream)
    splits = torch.linspace(0, n, P + 1, device="cuda").to(torch.int32)
    splits[-1] = n
    ws = torch.empty(lib.srj_kudo_workspace_bytes(len(cols), P), dtype=torch.uint8, device="cuda")
    offs = torch.empty(P + 1, dtype=torch.int64, device="cuda")
    total = ctypes.c_int64(0)
    cin = (N.SrjColumn * len(cols))(*[c._c() for c in cols])
    N.check(lib.srj_kudo_split_sizes(cin, len(cols), n, splits.data_ptr(), P, offs.data_ptr(), ctypes.byref(total), ws.data_ptr(), st))
    buf = torch.empty(total.value, dtype=torch.uint8, device="cuda")
    words = (n + 31) // 32
    outs = [S.ColumnVector(c.dtype, n, torch.empty_like(c.data), torch.empty(words, dtype=torch.int32, device="cuda")) for c in cols]
    cout = (N.SrjColumn * len(cols))(*[c._c() for c in outs])
    ids = (C_int32 * len(types))(*types)
    rows = ctypes.c_int64(0)
    chars = (ctypes.c_int64 * len(types))()

    def split():
        N.check(lib.srj_kudo_split(cin, len(cols), n, splits.data_ptr(), P, offs.data_ptr(), buf.data_ptr(), ws.data_ptr(), st))

    def assemble():
        N.check(lib.srj_kudo_assemble(buf.data_ptr(), offs.data_ptr(), P, cout, len(cols), n, ws.data_ptr(), st))

    split()
    N.check(lib.srj_kudo_assemble_sizes(buf.data_ptr(), offs.data_ptr(), P, ids, len(types), ctypes.byref(rows), chars, ws.data_ptr(), st))
    assert rows.value == n
    assemble()
    torch.cuda.synchronize()
    for i in (0, 9, 22):                                     # assemble(split(x)) = x: data and masks of three columns
        assert torch.equal(outs[i].data, cols[i].data) and torch.equal(outs[i].mask, cols[i].mask)
    step = assemble if args.direction == "from_rows" else split
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(0)
    sampler.start()
    stream = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    peak, peak_src = load_peaks()
    bpr = 2 * (sum(SIZE[t] for t in types) + len(types) / 8.0)     # the table once, the partitions once
    gbs = bpr * n / (ms * 1e-3) / 1e9
    what = "assemble" if args.direction == "from_rows" else "split"
    print(json.dumps({"metric": f"rows_per_sec_kudo_{what}", "value": n / (ms * 1e-3), "unit": "rows/s", "n_gpus": 1, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
                      "data": "synthetic", "config": {"workload": wl["name"], "rows": n, "partitions": P, "buffer_bytes": total.value,
                                                      "l2": "table 9.6 GB + buffer 9.9 GB >> 126 MB L2"},
                      "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": peak, "unit": "GB/s", "frac": round(gbs / peak, 4), "traffic": None,
                                   "kernel": f"kudo_{what}_kernel", "algorithmic_bytes_per_row": bpr, "peak_source": peak_src},
                      "cpu_baseline": _cpu_f("kudo_" + what, wl, 4_000_000, P=P), "e2e": None, "gpu_launches": args.steps, "clocks": clocks}))


def run_unsafe(args, wl, rank, world):
    """columns <-> UnsafeRow on one GPU, inputs resident in HBM; --direction picks the timed side."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "spark-rapids-jni_b200"))
    import srj_b200 as S
    from srj_b200 import _native as N
    torch.cuda.set_device(0)
    types, n = wl["types"], args.rows or wl["rows"]
    cols = synth_columns_gpu(torch, S, types, n, wl["null_frac"], 42)
    lib = N.lib()
    ids = (C_int32 * len(types))(*types)
    a, b = C_int32(0), C_int32(0)
    N.check(lib.srj_unsafe_row_layout(ids, len(types), ctypes.byref(a), ctypes.byref(b)))
    row_bytes = b.value
    st = int(torch.cuda.current_stream().cuda_stream)
    ws = torch.empty(lib.srj_unsafe_row_workspace_bytes(len(types), n), dtype=torch.uint8, device="cuda")
    rows = torch.empty(n * row_bytes, dtype=torch.uint8, device="cuda")
    words = (n + 31) // 32
    outs = [S.ColumnVector(c.dtype, n, torch.empty_like(c.data), torch.empty(words, dtype=torch.int32, device="cuda")) for c in cols]
    nulls = torch.zeros(len(cols), dtype=torch.int64, device="cuda")
    cin = (N.SrjColumn * len(cols))(*[c._c() for c in cols])
    cout = (N.SrjColumn * len(cols))(*[c._c() for c in outs])

    def to_rows():
        N.check(lib.srj_convert_to_unsafe_rows(cin, len(cols), n, None, rows.data_ptr(), ws.data_ptr(), st))

    def from_rows():
        N.check(lib.srj_convert_from_unsafe_rows(rows.data_ptr(), None, n, cout, len(cols), nulls.data_ptr(), ws.data_ptr(), st))

    to_rows()
    from_rows()
    torch.cuda.synchronize()
    # round trip identity on the valid values of two columns + the null counts
    for i in (3, 5):
        m = cols[i].mask
        valid = ((m[torch.arange(n, device="cuda") // 32] >> (torch.arange(n, device="cuda") % 32)) & 1).bool()
        assert torch.equal(outs[i].data.view(torch.int64)[valid], cols[i].data.view(torch.int64)[valid])
        assert int(nulls[i]) == int((~valid).sum())
    step = to_rows if args.direction == "to_rows" else from_rows
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(0)
    sampler.start()
    stream = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    peak, peak_src = load_peaks()
    bpr = row_bytes + sum(SIZE[t] for t in types) + len(types) / 8.0
    gbs = bpr * n / (ms * 1e-3) / 1e9
    print(json.dumps({"metric": f"rows_per_sec_convert_{'to' if args.direction == 'to_rows' else 'from'}_unsafe_rows", "value": n / (ms * 1e-3),
                      "unit": "rows/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                      "config": {"workload": wl["name"], "rows": n, "row_bytes": row_bytes, "direction": args.direction,
                                 "l2": "rows 13.2 GB + columns 7.2 GB >> 126 MB L2"},
                      "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": peak, "unit": "GB/s", "frac": round(gbs / peak, 4),
                                   "traffic": None, "kernel": "ur_to_rows_kernel" if args.direction == "to_rows" else "ur_from_rows_kernel",
                                   "algorithmic_bytes_per_row": bpr, "peak_source": peak_src},
                      "cpu_baseline": _cpu_f("unsafe_to" if args.direction == "to_rows" else "unsafe_from", wl, 2_000_000), "e2e": None, "gpu_launches": args.steps, "clocks": clocks}))


def run_reference(args, wl, rank, world):
    """--impl reference: the CPU implementation of the path on the host cores (oracle port: the reference's own
    code needs a JVM + libcudf, neither exists here).  Rank 0 only."""
    if rank != 0:
        return
    from oracle import oracle as O
    types = wl["types"]
    nthreads = os.cpu_count()
    if STRING in types:
        # C3: one batch of the workload generated on the host (to_rows by the threaded oracle: first touch of the row
        # buffer is spread over the cores), converted by the oracle's threaded from_rows; best of the steps
        nb = int(min(args.rows or wl["batch_rows"], wl["batch_rows"]))
        cols = synth_c3_host(types, nb, wl["null_frac"], seed=4242)
        rs = O.row_sizes(cols)
        offs = np.zeros(nb + 1, np.int32)
        np.cumsum(rs, out=offs[1:])
        rows = np.empty(int(offs[-1]), np.uint8)
        O.to_rows_mt(cols, 0, nb, offs, rows, nthreads)
        words = (nb + 31) // 32
        hc = [O.HCol(t, np.empty(max(len(c.data), 1), np.uint8), np.empty(words, np.uint32),
                     np.empty(nb + 1, np.int32) if t == STRING else None, 0, nb) for t, c in zip(types, cols)]
        for _ in range(max(1, args.warmup)):
            O.from_rows_mt(rows, offs, nb, hc, nthreads)
        assert np.array_equal(hc[3].offsets, cols[3].offsets) and np.array_equal(hc[0].data[: nb * 4], cols[0].data)
        times = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            O.from_rows_mt(rows, offs, nb, hc, nthreads)
            times.append(time.perf_counter() - t0)
        sec = float(np.mean(times))
        v = nb / sec
        cfg = {"workload": wl["name"], "direction": "from_rows", "rows_per_step": nb, "batch_rows": nb,
               "avg_row_bytes": len(rows) / nb, "columns": len(types)}
        cpu = {"value": v, "unit": "rows/s", "cores": nthreads, "kind": "port", "best": nb / min(times),
               "sample": f"one {nb}-row batch of the {wl['rows']}-row workload per step, {nthreads} OpenMP threads "
                         f"(oracle/srj_oracle.c orc_from_rows_mt)"}
    else:
        st, sz, voff, spr = O.compute_layout(types)
        row_size = (spr + 7) // 8 * 8
        n = int(min(args.rows or wl["rows"], args.cpu_sample_rows))
        data = np.empty(n * row_size, np.uint8)
        step_ = 1 << 26                                  # filled in pieces: any bytes are valid fixed-width JCUDF rows
        rng = np.random.Generator(np.random.Philox(42))
        for o in range(0, len(data), step_):
            data[o:o + step_] = rng.integers(0, 256, min(step_, len(data) - o), dtype=np.uint8)
        cols = [O.HCol(t, np.empty(n * SIZE[t], np.uint8), np.empty((n + 31) // 32, np.uint32), None, 0, n) for t in types]
        for _ in range(max(1, args.warmup)):
            O.from_rows_fixed_mt(data, n, cols, nthreads)
        times = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            O.from_rows_fixed_mt(data, n, cols, nthreads)
            times.append(time.perf_counter() - t0)
        sec = float(np.mean(times))
        v = n / sec
        cfg = {"workload": wl["name"], "rows_per_step": n, "row_bytes": row_size, "columns": len(types),
               "note": "row conversion only" + (" (the fused hash of the GPU arm is not part of this CPU loop)" if "hash_keys" in wl else "")}
        cpu = {"value": v, "unit": "rows/s", "cores": nthreads, "kind": "port", "best": n / min(times),
               "sample": f"{n} rows per step (bounded sample of the {wl['rows']}-row workload), {nthreads} OpenMP threads"}
    print(json.dumps({"impl": "reference", "metric": "rows_per_sec_convert_from_rows", "value": v, "unit": "rows/s",
                      "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
                      "higher_is_better": True, "scaling": "strong" if STRING in types else "weak", "vs_baseline": None,
                      "dtype": "u8", "data": "synthetic", "config": cfg, "cpu_baseline": cpu,
                      "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0,
                      "note": "CPU restatement of the reference algorithm (oracle port); the reference's CUDA path cannot be "
                              "built here (needs libcudf+rmm+JDK)"}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS),
                    help="c3 (default) = the configuration BASELINE.json's metric is quoted on; c2 / c4 = its other 1-GPU configs")
    ap.add_argument("--rows", type=int, default=0, help="override rows per GPU (development only)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-sample-rows", type=int, default=16_000_000)
    ap.add_argument("--direction", default="from_rows", choices=["from_rows", "to_rows"])  # kudo: to_rows = split, from_rows = assemble
    ap.add_argument("--no-gather", action="store_true", help="multi-GPU: skip the all-gather (conversion-only scaling)")
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"],
                    help="multi-GPU all-gather transport: copy engines over NVLink peer memory (default) or ncclAllGather")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="c3: after the timed steps, write a fixed seeded sample of what the last step computed as DIR/<name>.npy "
                         "(rank 0; same arguments give the same inputs, so two builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c3"):
        ap.error("--dump-outputs is implemented for --workload c3 --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
    elif wl.get("nvbench"):
        if rank == 0:
            run_nvbench(args, wl, rank, world)
    elif wl.get("partition"):
        if rank == 0:
            run_partition(args, wl, rank, world)
    elif wl.get("shuffle"):
        run_shuffle(args, wl, rank, world)
    elif wl.get("kudo"):
        if rank == 0:
            run_kudo(args, wl, rank, world)
    elif wl.get("unsafe"):
        if rank == 0:
            run_unsafe(args, wl, rank, world)
    elif args.workload == "c3":
        run_c3(args, wl, rank, world)
    else:
        run_ours(args, wl, rank, world)


if __name__ == "__main__":
    main()
