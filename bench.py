#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Spark SQL hot path (BASELINE.json: "TPC-H Q1/Q3/Q5 rows/sec at
SF100, 1/2/4/8 B200; op HBM GB/s vs 8 TB/s").

One process per GPU.  Every rank owns one SF100-shaped shard of the synthetic TPC-H dataset (include/sb_synth.h, generated
on the device by sb_synth_table with seed 42 + rank: 150 M orders, 599,999,994 lineitem rows) -- weak scaling, the database
grows with the number of GPUs and is partitioned by order, so every join is shard-local (customer / supplier / nation /
region are replicated like broadcast relations) and shards meet only where the plan has an exchange:
  Q1  HashAggregate(partial, Filter+Project fused) -> [SinglePartition exchange = sb_all_gather] -> HashAggregate(final) -> Sort
  Q3  2 x BroadcastHashJoin -> HashAggregate -> TakeOrderedAndProject(10) -> [all_gather of the 10 rows] -> TakeOrdered(10)
  Q5  5 joins -> HashAggregate(partial) -> [all_gather] -> HashAggregate(final) -> Sort
  shuffle (N > 1 only; BASELINE.json configs[3] shape: 74 B/row lineitem rows, HashPartitioning(l_orderkey, 2048)):
      sb_hash_partition (Murmur3 pmod ids + stable multisplit) -> sb_all_to_all over NVLink.

The ONE JSON line on stdout (rank 0) is the Q1 leg (`metric` tpch_q1_rows_per_sec, `config.workload` names it); `legs`
carries the same fields for q3, q5 and (N > 1) shuffle.  Per leg:
  value      lineitem rows / s with the columns already resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e        the same plan through the public operator API from HOST buffers: H2D inside the timed region, result read back.
             Q1 reads Parquet-style encoded column chunks (dictionary + RLE/bit-packed pages, PLAIN doubles) and decodes them
             on the GPU (sb_scan_decode) row group by row group into the streaming aggregate (sb_hash_agg_update) -- the plain
             38 B/row variant is reported next to it; Q3/Q5 import plain pinned columns.  h2d_bytes_per_step counts what
             actually crossed PCIe.
  roofline   dominant kernel: algorithmic bytes (SURVEY.md 8d) / its CUDA-event time (sb_profile_*) vs MEASURED_PEAKS.json
  verified   the GPU result of the measured run equals the CPU oracle's answer on the same rows (keys / counts / order exact,
             floating sums 1e-6 relative); N > 1: checked per rank before the exchange-level merge, and the merged result
             against the merge of the oracle answers.
`--impl reference` times the reference's CPU path (the oracle's whole-stage restatements, kind "port": the reference is
JVM-only and this image has no JDK) on the host cores the cgroup grants, on the same rows.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ORDERS_PER_SF = 1_500_000
NATION_REGION = [0, 1, 1, 1, 4, 0, 3, 3, 2, 2, 4, 4, 2, 4, 0, 0, 0, 1, 2, 3, 4, 2, 3, 3, 1]


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"     # B200_PROFILING.md fallback


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed regions (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # median over the samples taken under load (the sampler also sees the idle gaps between legs)
        busy = [x for x in sm if smax and x >= 0.5 * max(smax)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------- host CPU side
def ncu_traffic(kernel, rows):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel` from the committed `ncu --set full` capture of this
    workload (profiles/r02_ncu_traffic.json, written from the capture by tools/ncu_traffic.py); null when the capture was taken at
    another size (a profiler cannot run inside the timed region)."""
    try:
        rec = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r02_ncu_traffic.json")))[kernel]
    except Exception:
        return {"traffic": None, "traffic_note": "no ncu capture committed for this kernel"}
    if int(rec.get("rows", -1)) != int(rows):
        return {"traffic": None, "traffic_note": "the committed ncu capture (%s) is for %s rows per launch, this run has %d"
                % (rec.get("source"), rec.get("rows"), rows)}
    return {"traffic": int(rec["dram_bytes"]), "traffic_note": "from %s" % rec.get("source")}


def host_threads(share=1):
    """Threads the CPU arm may really use: the affinity mask capped by this process's share (1 / share) of the cgroup's CPU quota (cpu.max)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(math.ceil(int(quota) / int(period))) // share))
    except Exception:
        pass
    return n


def rank_cpu_block(cpus, local_rank, world):
    """The block of host CPUs rank `local_rank` of `world` ranks on one host keeps: contiguous, disjoint, equal-sized (the remainder
    stays unused).  [] when there are fewer CPUs than ranks (the mask is then left alone)."""
    cpus = sorted(cpus)
    per = len(cpus) // world
    return cpus[local_rank * per:(local_rank + 1) * per] if per >= 1 else []


def _omp_setup(share=1):
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every thread the cgroup grants, spread over the sockets."""
    nt = host_threads(share)
    os.environ["OMP_NUM_THREADS"] = str(nt)
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "cores")
    return nt


class HostData:
    """The rank's shard on the host, filled by the oracle's OpenMP generator (parallel first touch: pages land on the NUMA
    node of the thread that scans them in the baseline loops).  CPU legs only."""

    def __init__(self, n_orders, seed, tables):
        from oracle import tpch_oracle as TO
        from spark_b200 import tpch
        self.n_orders = n_orders
        self.cols = {}
        for table, columns in tables.items():
            self.cols.update(TO.synth_host(table, columns, n_orders, seed))
        self.n_li = tpch.synth_rows("lineitem", n_orders)
        self.n_ord = n_orders
        self.n_cust = tpch.synth_rows("customer", n_orders)
        self.n_supp = tpch.synth_rows("supplier", n_orders)


def cpu_q1(h: HostData):
    from oracle import oracle as O
    from spark_b200 import tpch
    L = O.lib()
    k0 = np.zeros(16, np.int8); k1 = np.zeros(16, np.int8); sums = np.zeros(80); cnt = np.zeros(16, np.int64)
    c = h.cols
    t0 = time.perf_counter()
    ng = L.so_q1_partial_final(c["l_quantity"].ctypes.data, c["l_extendedprice"].ctypes.data, c["l_discount"].ctypes.data,
                               c["l_tax"].ctypes.data, c["l_returnflag"].ctypes.data, c["l_linestatus"].ctypes.data,
                               c["l_shipdate"].ctypes.data, h.n_li, tpch.Q1_CUTOFF, 16, k0.ctypes.data, k1.ctypes.data,
                               sums.ctypes.data, cnt.ctypes.data)
    dt = time.perf_counter() - t0
    rows = sorted((int(k0[g]), int(k1[g]), [float(x) for x in sums[g * 5:g * 5 + 5]], int(cnt[g])) for g in range(ng))
    return dt, rows


def cpu_q3(h: HostData):
    from oracle import oracle as O
    from spark_b200 import tpch
    L = O.lib()
    c = h.cols
    ok = np.zeros(10, np.int64); rev = np.zeros(10); od = np.zeros(10, np.int32); sp = np.zeros(10, np.int32); groups = C.c_int64()
    t0 = time.perf_counter()
    n = L.so_q3(c["c_custkey"].ctypes.data, c["c_mktsegment"].ctypes.data, h.n_cust,
                c["o_orderkey"].ctypes.data, c["o_custkey"].ctypes.data, c["o_orderdate"].ctypes.data, c["o_shippriority"].ctypes.data, h.n_ord,
                c["l_orderkey"].ctypes.data, c["l_extendedprice"].ctypes.data, c["l_discount"].ctypes.data, c["l_shipdate"].ctypes.data, h.n_li,
                tpch.Q3_SEGMENT, tpch.Q3_DATE, 10, ok.ctypes.data, rev.ctypes.data, od.ctypes.data, sp.ctypes.data, C.byref(groups))
    dt = time.perf_counter() - t0
    return dt, [(int(ok[i]), float(rev[i]), int(od[i]), int(sp[i])) for i in range(n)]


def cpu_q5(h: HostData):
    from oracle import oracle as O
    from spark_b200 import tpch
    L = O.lib()
    c = h.cols
    nr = np.array(NATION_REGION, np.int32); rev = np.zeros(25); seen = np.zeros(25, np.uint8)
    t0 = time.perf_counter()
    L.so_q5(c["c_custkey"].ctypes.data, c["c_nationkey"].ctypes.data, h.n_cust,
            c["o_orderkey"].ctypes.data, c["o_custkey"].ctypes.data, c["o_orderdate"].ctypes.data, h.n_ord,
            c["l_orderkey"].ctypes.data, c["l_suppkey"].ctypes.data, c["l_extendedprice"].ctypes.data, c["l_discount"].ctypes.data, h.n_li,
            c["s_suppkey"].ctypes.data, c["s_nationkey"].ctypes.data, h.n_supp,
            nr.ctypes.data, tpch.Q5_REGION, tpch.Q5_DATE_LO, tpch.Q5_DATE_HI, rev.ctypes.data, seen.ctypes.data)
    dt = time.perf_counter() - t0
    rows = sorted(((int(g), float(rev[g])) for g in range(25) if seen[g]), key=lambda r: -r[1])
    return dt, rows


CPU_TABLES = {
    "q1": {"lineitem": ["l_quantity", "l_extendedprice", "l_discount", "l_tax", "l_returnflag", "l_linestatus", "l_shipdate"]},
    "q3": {"lineitem": ["l_orderkey", "l_extendedprice", "l_discount", "l_shipdate"],
           "orders": ["o_orderkey", "o_custkey", "o_orderdate", "o_shippriority"], "customer": ["c_custkey", "c_mktsegment"]},
    "q5": {"lineitem": ["l_orderkey", "l_suppkey", "l_extendedprice", "l_discount"], "orders": ["o_orderkey", "o_custkey", "o_orderdate"],
           "customer": ["c_custkey", "c_nationkey"], "supplier": ["s_suppkey", "s_nationkey"]},
}
CPU_FN = {"q1": cpu_q1, "q3": cpu_q3, "q5": cpu_q5}


def _close(a, b, rtol=1e-6):
    return abs(a - b) <= rtol * max(abs(a), abs(b), 1e-300)


def check_q1(gpu_rows, cpu_rows):
    """gpu_rows / cpu_rows: sorted [(flag, status, [sum_qty, sum_price, sum_disc_price, sum_charge, sum_disc], count)]"""
    if len(gpu_rows) != len(cpu_rows):
        return False
    for g, c in zip(gpu_rows, cpu_rows):
        if g[0] != c[0] or g[1] != c[1] or g[3] != c[3]:
            return False
        if not all(_close(x, y) for x, y in zip(g[2], c[2])):
            return False
    return True


def check_q3(gpu_rows, cpu_rows):
    if len(gpu_rows) != len(cpu_rows):
        return False
    for g, c in zip(gpu_rows, cpu_rows):       # ORDER BY revenue DESC, o_orderdate: order is part of the answer
        if g[0] != c[0] or g[2] != c[2] or g[3] != c[3] or not _close(g[1], c[1]):
            return False
    return True


def check_q5(gpu_rows, cpu_rows):
    if len(gpu_rows) != len(cpu_rows):
        return False
    return all(g[0] == c[0] and _close(g[1], c[1]) for g, c in zip(gpu_rows, cpu_rows))


def dump_outputs(out_dir, results):
    """results: leg -> pyarrow.Table.  One float64 array per column (dates as days since the epoch, NULL as NaN); the query
    results are at most a few dozen rows, far below any size worth sampling."""
    import pyarrow as pa
    os.makedirs(out_dir, exist_ok=True)
    for leg, tbl in results.items():
        for name in tbl.column_names:
            col = tbl.column(name)
            if pa.types.is_date(col.type):
                col = col.cast(pa.int32())
            np.save(os.path.join(out_dir, "%s_%s.npy" % (leg, name)), col.cast(pa.float64()).to_numpy())


def run_reference(args, rank):
    """--impl reference: the reference's CPU path (oracle port) on the same rows, host cores only; rank 0 alone works."""
    if rank != 0:
        return
    nt = _omp_setup()
    from oracle import oracle as O
    O.lib().so_set_threads(nt)
    n_orders = int(ORDERS_PER_SF * args.sf)
    legs = {}
    line = None
    for leg in args.legs:
        if leg == "shuffle":
            continue
        t0 = time.perf_counter()
        h = HostData(n_orders, 42, CPU_TABLES[leg])
        gen_s = time.perf_counter() - t0
        steps = args.steps if leg == "q1" else max(1, min(args.steps, args.leg_steps))
        warm = args.warmup if leg == "q1" else min(args.warmup, 1)
        times = [CPU_FN[leg](h)[0] for _ in range(warm + steps)][warm:]
        ms = 1000.0 * sum(times) / len(times)
        value = h.n_li / (ms / 1000.0)
        d = {"value": value, "unit": "rows/s", "ms_per_step": ms, "steps": steps, "rows": h.n_li, "datagen_s": gen_s}
        legs[leg] = d
        del h
    q1 = legs.get("q1") or next(iter(legs.values()))
    line = {"impl": "reference", "metric": "tpch_q1_rows_per_sec", "value": q1["value"], "unit": "rows/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": q1["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "TPC-H Q1 SF%g (scan+filter+hash-agg on lineitem), CPU whole-stage restatement, decoded columns in host DRAM" % args.sf,
                       "rows": q1["rows"], "bytes_per_row": 38},
            "cpu_baseline": {"value": q1["value"], "unit": "rows/s", "cores": nt, "kind": "port",
                             "sample": "full SF%g lineitem (%d rows) per step; OpenMP static loops, parallel first touch, OMP_PROC_BIND=%s"
                                       % (args.sf, q1["rows"], os.environ.get("OMP_PROC_BIND")),
                             "host_read_gbs": q1["rows"] * 38 / (q1["ms_per_step"] / 1000.0) / 1e9},
            "e2e": {"value": q1["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "legs": legs, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sf", type=float, default=100.0, help="TPC-H scale factor per GPU (default 100 = the configuration the metric is quoted on)")
    ap.add_argument("--legs", default="q1,q3,q5,shuffle", help="comma list of q1,q3,q5,shuffle (shuffle runs only with --gpus > 1)")
    ap.add_argument("--leg-steps", type=int, default=5, help="timed steps of the q3 / q5 / shuffle legs")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--shuffle-rows", type=int, default=96_000_000, help="rows per GPU of the shuffle leg (74 B/row)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--profile-host", action="store_true", help="cProfile one untimed step of every join leg to stderr (debugging)")
    ap.add_argument("--config", action="append", default=[], metavar="KEY=VALUE", help="sb_config_set(KEY, VALUE) before the run (A/B experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of the last timed step of every query leg to DIR/<leg>_<column>.npy "
                                                          "(float64), to compare two builds output for output")
    args = ap.parse_args()
    args.legs = [x for x in args.legs.split(",") if x]
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world == 1:
        args.legs = [x for x in args.legs if x != "shuffle"]
    partitioned = False
    if world > 1:
        # One rank per GPU on ONE host: give every rank its own block of the CPUs the job may use, before any OpenMP runtime loads.
        # With OMP_PROC_BIND every rank's master thread is bound to the FIRST place of its mask -- with a shared mask that is the same
        # core for all ranks, and the host threads (which spin in cudaStreamSynchronize between operators) then time-slice it: measured
        # at N = 4 before this fix, Q1 took 18 ms per step with 4.3 ms of kernels (gpurun_out r26 -> profiles/r02_bench_n4_shared_mask.json).
        try:
            mine = rank_cpu_block(os.sched_getaffinity(0), local_rank, world)
            if mine:
                os.sched_setaffinity(0, mine)
                partitioned = True
        except (AttributeError, OSError):
            pass
    nt = _omp_setup(world)             # before any OpenMP runtime is loaded; every rank checks its own shard against the oracle at the same time
    if world > 1 and not partitioned:  # shared mask: at least do not oversubscribe it
        nt = max(1, min(nt, len(os.sched_getaffinity(0)) // world))
        os.environ["OMP_NUM_THREADS"] = str(nt)

    import pyarrow as pa
    import torch
    import torch.distributed as dist
    from spark_b200 import _capi as capi, tpch
    from spark_b200.columnar import ColumnarBatch, HostColumn, PinnedArray, Stream
    from spark_b200.execution import (BroadcastHashJoinExec, HashAggregateExec, HashPartitioning, LocalTableScanExec, ShuffleExchangeExec,
                                      SortExec, SparkPlan, TakeOrderedAndProjectExec)
    from spark_b200.expressions import SortOrder

    lib = capi.init(local_rank)
    for kv in args.config:
        k, v = kv.split("=", 1)
        capi.config_set(k, int(v))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        idbuf = torch.zeros(capi.SB_UNIQUE_ID_BYTES, dtype=torch.uint8, device="cuda")
        if rank == 0:
            raw = C.create_string_buffer(capi.SB_UNIQUE_ID_BYTES)
            capi.check(lib.sb_comm_get_unique_id(raw))
            idbuf.copy_(torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8))
        dist.broadcast(idbuf, 0)
        capi.check(lib.sb_comm_init(rank, world, bytes(idbuf.cpu().numpy().tobytes())))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_true(ok):
        if world == 1:
            return bool(ok)
        t = torch.tensor([1 if ok else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    stream = Stream()
    peak, peak_src = _peaks()
    n_orders = int(ORDERS_PER_SF * args.sf)
    seed = 42 + rank
    n_li = tpch.synth_rows("lineitem", n_orders)

    class AllGatherExec(SparkPlan):
        """SinglePartition / broadcast exchange of a small table: every rank receives all ranks' rows (sb_all_gather)."""

        def __init__(self, child):
            self.child = child

        def executeColumnar(self, stream=None):
            inp = self.child.executeColumnar(stream)
            if world == 1:
                return inp
            try:
                h = C.c_void_p()
                capi.check(lib.sb_all_gather(inp.handle, stream.handle, C.byref(h)))
                return ColumnarBatch(h, inp.names, inp.arrow_types)
            finally:
                inp.close()

    class BatchSource(SparkPlan):
        """Leaf whose batch is swapped per step, so the operator tree (and its compiled plans) is built once."""

        def __init__(self, batch=None):
            self.batch = batch

        def executeColumnar(self, stream=None):
            return self.batch.rename(self.batch.names)

    # ---- resident tables ------------------------------------------------------------------------------------------------
    li_cols = ["l_orderkey", "l_suppkey", "l_quantity", "l_extendedprice", "l_discount", "l_tax", "l_returnflag", "l_linestatus", "l_shipdate"]
    need_join = any(x in args.legs for x in ("q3", "q5"))
    if not need_join:
        li_cols = tpch.Q1_COLUMNS
    lineitem = tpch.synth_batch("lineitem", li_cols, n_orders, seed, stream=stream)
    tables = {"lineitem": lineitem}
    if need_join:
        tables["orders"] = tpch.synth_batch("orders", tpch.SYNTH_COLUMNS["orders"], n_orders, seed, stream=stream)
        tables["customer"] = tpch.synth_batch("customer", tpch.SYNTH_COLUMNS["customer"], n_orders, seed, stream=stream)
        tables["supplier"] = tpch.synth_batch("supplier", tpch.SYNTH_COLUMNS["supplier"], n_orders, seed, stream=stream)
        tables["nation"] = ColumnarBatch.from_arrow(tpch.nation_table(), stream)
        tables["region"] = ColumnarBatch.from_arrow(tpch.region_table(), stream)
    stream.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    def time_resident(step, steps, warmup, kernel_names=()):
        for _ in range(warmup):
            step()
        capi.check(lib.sb_profile_enable(1))
        capi.check(lib.sb_profile_reset())
        barrier()
        l0 = capi.kernel_launch_count()
        total_ms, per_step = 0.0, []
        for _ in range(steps):                           # CUDA events on the operators' stream around every step
            stream.record_start()
            step()
            stream.record_stop()
            per_step.append(stream.elapsed_ms())
            total_ms += per_step[-1]
        barrier()
        launches = capi.kernel_launch_count() - l0
        prof = capi.profile_dump()                       # every device-timed section of the library
        for k in kernel_names:
            prof.setdefault(k, (0.0, 0))
        capi.check(lib.sb_profile_enable(0))
        last_step_ms[:] = per_step
        return max_over_ranks(total_ms / steps), launches, prof

    last_step_ms = []

    def time_e2e(step, steps):
        step()          # warm-up (allocator pools, compiled plans)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = step()
        stream.synchronize()
        ms = 1000.0 * (time.perf_counter() - t0) / steps
        barrier()
        return max_over_ranks(ms), res

    legs = {}
    cpu_info = None
    # A timed step keeps the batch it returns until the leg's next step starts (the same one release per step as closing it at
    # once), so the last timed step's result is still there for --dump-outputs.
    held = {}
    results = {}

    def release_held(leg):
        b = held.pop(leg, None)
        if b is not None:
            b.close()

    def take_result(leg):
        if args.dump_outputs:
            results[leg] = held[leg].to_arrow(stream)
        release_held(leg)

    def cpu_leg(leg):
        """Oracle answer for this rank's shard (verification) and, at N = 1 on rank 0, the timed CPU baseline."""
        if args.no_verify and (args.no_cpu_baseline or world > 1):
            return None, None
        from oracle import oracle as O
        O.lib().so_set_threads(nt)
        h = HostData(n_orders, seed, CPU_TABLES[leg])
        dt, rows = CPU_FN[leg](h)                 # first pass: answer (and warm-up)
        timing = None
        if world == 1 and not args.no_cpu_baseline:
            reps = 6 if leg == "q1" else 2
            ts = [CPU_FN[leg](h)[0] for _ in range(reps)]
            mean = sum(ts) / len(ts)
            timing = {"value": h.n_li / mean, "unit": "rows/s", "cores": nt, "kind": "port",
                      "sample": "full SF%g shard (%d lineitem rows) x %d passes after 1 warm-up, mean; %.1f core-seconds; OpenMP, parallel "
                                "first touch, OMP_PROC_BIND=%s" % (args.sf, h.n_li, reps, sum(ts) * nt, os.environ.get("OMP_PROC_BIND"))}
        del h
        return rows, timing

    # ===================================================================================================== Q1
    if "q1" in args.legs:
        q1_src = BatchSource(lineitem.select(tpch.Q1_COLUMNS))
        partial = tpch.q1_partial_plan(q1_src, fused=True)
        q1_plan = tpch.q1_final_plan(AllGatherExec(partial), sort=True)

        def q1_rows(tbl):
            """pyarrow result -> [(flag, status, [sum_qty, sum_price, sum_disc_price, sum_charge, sum_disc], count)]"""
            cols = {n: tbl.column(n).to_pylist() for n in tbl.column_names}
            out = []
            for i in range(tbl.num_rows):
                cnt = cols["count_order"][i]
                out.append((cols["l_returnflag"][i], cols["l_linestatus"][i],
                            [cols["sum_qty"][i], cols["sum_base_price"][i], cols["sum_disc_price"][i], cols["sum_charge"][i],
                             cols["avg_disc"][i] * cnt], cnt))
            return out

        def step_q1():
            release_held("q1")
            held["q1"] = q1_plan.executeColumnar(stream)

        ms, launches, prof = time_resident(step_q1, args.steps, args.warmup, ("agg_update",))
        take_result("q1")
        plan_name = lib.sb_hash_aggregate_last_plan().decode()
        # which kernels ran the big launch: run the Partial stage once more and ask
        p_once = partial.executeColumnar(stream); p_once.close()
        plan_name = lib.sb_hash_aggregate_last_plan().decode()
        kernel_ms = prof["agg_update"][0] / max(1, args.steps)
        alg_bytes = n_li * tpch.Q1_BYTES_PER_ROW
        achieved = alg_bytes / (kernel_ms / 1000.0) / 1e9 if kernel_ms > 0 else 0.0
        # per-rank verification against the oracle, BEFORE the exchange-level merge
        gpu_local = tpch.q1_final_plan(partial, sort=True).collect(stream)
        verified = None
        cpu_rows, cpu_t = cpu_leg("q1")
        if cpu_rows is not None:
            verified = all_true(check_q1(q1_rows(gpu_local), cpu_rows))
        if world == 1:
            cpu_info = cpu_t
        # the generic kernels (no run-time specialisation) and a nullable / reordered variant of the same query, for the record
        variants = {}
        capi.config_set("agg_rtc", 0)
        v_ms, _, v_prof = time_resident(step_q1, max(3, args.steps // 4), 1, ("agg_update",))
        variants["generic_kernels"] = {"ms_per_step": v_ms, "agg_update_ms": v_prof["agg_update"][0] / max(1, max(3, args.steps // 4))}
        release_held("q1")
        capi.config_set("agg_rtc", 1)
        # the same query over NULLable columns handed over in another order (what a Parquet scan of a nullable schema gives Spark).
        # (a) the batch declares null_count = 0 (ColumnVector.hasNull() == false): the bitmaps are never read, same kernels as the
        #     headline; (b) null_count unknown: every referenced column's validity bitmap is read (another PlanMeta, specialised at
        #     run time like any plan)
        order = ["l_shipdate", "l_tax", "l_linestatus", "l_discount", "l_returnflag", "l_extendedprice", "l_quantity"]
        ones = torch.full(((n_li + 7) // 8 + 64,), 255, dtype=torch.uint8, device="cuda")
        vsteps = max(3, args.steps // 4)
        for vname, null_count in (("nullable_schema_no_nulls_reordered", 0), ("nullable_columns_bitmaps_read_reordered", -1)):
            descs = (capi.sb_column * len(order))()
            for i, name in enumerate(order):
                descs[i] = lineitem.column_desc(lineitem.column_index(name))
                descs[i].validity = ones.data_ptr()
                descs[i].null_count = null_count
            hN = C.c_void_p()
            capi.check(lib.sb_table_import_device(descs, len(order), C.byref(hN)))
            nullable = ColumnarBatch(hN, order, [lineitem.arrow_types[lineitem.column_index(c)] for c in order])
            partial_n = tpch.q1_partial_plan(BatchSource(nullable), fused=True)
            q1n_plan = tpch.q1_final_plan(AllGatherExec(partial_n), sort=True)

            def step_q1n():
                out = q1n_plan.executeColumnar(stream)
                out.close()
            n_ms, _, n_prof = time_resident(step_q1n, vsteps, 2, ("agg_update",))
            p_once = partial_n.executeColumnar(stream); p_once.close()
            n_name = lib.sb_hash_aggregate_last_plan().decode()
            n_kernel = n_prof["agg_update"][0] / vsteps
            n_bytes = n_li * (tpch.Q1_BYTES_PER_ROW + (7.0 / 8.0 if null_count else 0.0))
            same = check_q1(q1_rows(q1n_plan.collect(stream)), q1_rows(q1_plan.collect(stream))) if world == 1 else None
            variants[vname] = {"ms_per_step": n_ms, "agg_update_ms": n_kernel, "agg_kernels": n_name,
                               "achieved_gbs": n_bytes / (n_kernel / 1000.0) / 1e9 if n_kernel else None,
                               "frac": n_bytes / (n_kernel / 1000.0) / 1e9 / peak if n_kernel else None,
                               "bytes_per_row": n_bytes / n_li, "equals_headline_result": same}
            nullable.close()
        del ones
        legs["q1"] = {"value": world * n_li / (ms / 1000.0), "unit": "rows/s", "ms_per_step": ms, "steps": args.steps, "rows_per_gpu": n_li,
                      "gpu_launches": int(launches), "verified": verified, "agg_kernels": plan_name, "variants": variants,
                      "roofline": {"bound": "hbm", "kernel": "agg_update_kernel (%s)" % plan_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                                   "frac": achieved / peak, "frac_of_8tbs_nominal": achieved / 8000.0, "peak_source": peak_src,
                                   "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": alg_bytes, **ncu_traffic("agg_update_kernel", n_li)}}

    # ===================================================================================================== Q3 / Q5
    def q3_rows(tbl):
        c = {n: tbl.column(n).to_pylist() for n in tbl.column_names}
        import datetime
        return [(c["l_orderkey"][i], c["revenue"][i], (c["o_orderdate"][i] - datetime.date(1970, 1, 1)).days, c["o_shippriority"][i])
                for i in range(tbl.num_rows)]

    def q5_rows(tbl):
        c = {n: tbl.column(n).to_pylist() for n in tbl.column_names}
        return [(c["n_name"][i], c["revenue"][i]) for i in range(tbl.num_rows)]

    def build_q3(src):
        local = tpch.q3_plan(src["customer"], src["orders"], src["lineitem"])
        if world == 1:
            return local, local
        merged = TakeOrderedAndProjectExec(10, [SortOrder("revenue", False), SortOrder("o_orderdate", True)], None, AllGatherExec(local))
        return local, merged

    def build_q5(src):
        # local = Partial -> Final on the shard; across shards the Partial rows meet through the all-gather
        full = tpch.q5_plan(src["customer"], src["orders"], src["lineitem"], src["supplier"], src["nation"], src["region"])
        if world == 1:
            return full, full
        part = full.child.child      # SortExec(Final(Partial(...)))
        aggs = full.child.aggregateExpressions
        merged = SortExec([("revenue", False, False)], HashAggregateExec(["n_name"], aggs, AllGatherExec(part), mode="final"))
        return full, merged

    join_legs = {"q3": (build_q3, q3_rows, check_q3,
                        {"lineitem": ["l_orderkey", "l_extendedprice", "l_discount", "l_shipdate"],
                         "orders": ["o_orderkey", "o_custkey", "o_orderdate", "o_shippriority"], "customer": ["c_custkey", "c_mktsegment"]}),
                 "q5": (build_q5, q5_rows, check_q5,
                        {"lineitem": ["l_orderkey", "l_suppkey", "l_extendedprice", "l_discount"], "orders": ["o_orderkey", "o_custkey", "o_orderdate"],
                         "customer": ["c_custkey", "c_nationkey"], "supplier": ["s_suppkey", "s_nationkey"]})}
    for leg in ("q3", "q5"):
        if leg not in args.legs:
            continue
        build, to_rows, check, used = join_legs[leg]
        src = {name: BatchSource(tables[name].select(cols)) for name, cols in used.items()}
        for small in ("nation", "region"):
            src[small] = BatchSource(tables[small])
        local_plan, merged_plan = build(src)

        def step_join():
            release_held(leg)
            held[leg] = merged_plan.executeColumnar(stream)

        steps = max(1, min(args.steps, args.leg_steps))
        if args.profile_host and rank == 0:
            import cProfile
            import pstats
            step_join()
            pr = cProfile.Profile()
            pr.enable()
            step_join()
            stream.synchronize()
            pr.disable()
            pstats.Stats(pr, stream=sys.stderr).sort_stats("cumulative").print_stats(25)
        ms, launches, prof = time_resident(step_join, steps, max(3, args.warmup), ("join_build", "join_probe", "join_fill", "gather", "filter_project", "agg_update"))
        take_result(leg)
        alg_bytes = sum(tpch.synth_rows(t, n_orders) * sum(tpch.synth_width(c) for c in cols) for t, cols in used.items())
        achieved = alg_bytes / (ms / 1000.0) / 1e9
        verified = None
        cpu_rows, cpu_t = cpu_leg(leg)
        if cpu_rows is not None:
            verified = all_true(check(to_rows(local_plan.collect(stream)), cpu_rows))
        # end to end: every referenced column crosses PCIe from pinned host buffers, then the plan, then the result comes back
        pinned = {}
        for t, cols in used.items():
            b = tables[t]
            for c in cols:
                pa_ = PinnedArray(b.num_rows, tpch.synth_dtype(c))
                capi.check(lib.sb_table_export_host(b.handle, b.column_index(c), pa_.array.ctypes.data, None, None, None, stream.handle))
                pinned[c] = pa_
        stream.synchronize()
        sbt = {np.dtype(np.int64): capi.SB_INT64, np.dtype(np.int32): capi.SB_INT32, np.dtype(np.int8): capi.SB_INT8, np.dtype(np.float64): capi.SB_FLOAT64}
        h2d = sum(p.nbytes for p in pinned.values())

        def step_e2e():
            fresh = {}
            for t, cols in used.items():
                hc = [HostColumn(capi.SB_DATE32 if c in tpch._DATE_COLS else sbt[pinned[c].dtype], pinned[c].array) for c in cols]
                fresh[t] = ColumnarBatch.from_host_columns(cols, hc, stream, [tables[t].arrow_types[tables[t].column_index(c)] for c in cols])
            for t, b in fresh.items():
                src[t].batch = b
            try:
                return merged_plan.collect(stream)
            finally:
                for t, b in fresh.items():
                    b.close()
                    src[t].batch = tables[t].select(used[t])

        e2e_ms, res = time_e2e(step_e2e, max(1, args.e2e_steps))
        d2h = int(sum(res.column(i).nbytes for i in range(res.num_columns)))
        for p in pinned.values():
            p.close()
        legs[leg] = {"value": world * n_li / (ms / 1000.0), "unit": "rows/s", "ms_per_step": ms, "steps": steps, "rows_per_gpu": n_li,
                     "gpu_launches": int(launches), "verified": verified, "step_ms": [round(x, 3) for x in last_step_ms],
                     "kernel_ms_per_step": {k: v[0] / steps for k, v in prof.items()},
                     "roofline": {"bound": "hbm", "kernel": "whole plan (sum of operator algorithmic bytes, SURVEY.md 8d: one read of every referenced column)",
                                  "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_of_8tbs_nominal": achieved / 8000.0,
                                  "peak_source": peak_src, "algorithmic_bytes_per_step": alg_bytes, "traffic": None},
                     "e2e": {"value": world * n_li / (e2e_ms / 1000.0), "unit": "rows/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                             "d2h_bytes_per_step": d2h, "input": "plain pinned host columns"},
                     "cpu_baseline": cpu_t}

    # ===================================================================================================== Q1 end to end (scan boundary)
    if "q1" in args.legs:
        e2e = run_q1_e2e(args, lib, capi, tpch, stream, lineitem, n_li, world, barrier, max_over_ranks, time_e2e, AllGatherExec, q1_rows, legs)
        legs["q1"]["e2e"] = e2e

    # ===================================================================================================== shuffle leg (N > 1)
    if "shuffle" in args.legs and world > 1:
        legs["shuffle"] = run_shuffle(args, lib, capi, tpch, stream, rank, world, n_orders, seed, barrier, max_over_ranks, all_true, time_resident, peak, peak_src)

    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        head = legs.get("q1") or next(iter(legs.values()))
        head_name = "q1" if "q1" in legs else next(iter(legs))
        line = {"metric": "tpch_%s_rows_per_sec" % head_name, "value": head["value"], "unit": "rows/s", "n_gpus": world, "steps": head["steps"],
                "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "TPC-H %s SF%g per GPU (%d lineitem rows; legs: %s)" % (head_name.upper(), args.sf, n_li, ",".join(legs)),
                           "rows_per_gpu": n_li, "bytes_per_row": tpch.Q1_BYTES_PER_ROW,
                           "plan": "HashAggregate(partial, fused Filter/Project)" + (" -> AllGather" if world > 1 else "") + " -> HashAggregate(final) -> Sort",
                           "l2_policy": "inputs (%.1f GB) larger than L2, no flush" % (n_li * tpch.Q1_BYTES_PER_ROW / 1e9),
                           "dataset": "include/sb_synth.h, seed 42 + rank, generated on the device"},
                "roofline": head.get("roofline"), "cpu_baseline": cpu_info, "e2e": head.get("e2e"), "verified": all(l.get("verified") is not False for l in legs.values()) and any(l.get("verified") for l in legs.values()),
                "gpu_launches": int(sum(l.get("gpu_launches", 0) for l in legs.values())), "legs": legs, "clocks": clocks}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, results)
        print(json.dumps(line), flush=True)
    for b in tables.values():
        b.close()
    if world > 1:
        capi.check(lib.sb_comm_destroy())
        dist.destroy_process_group()


def run_q1_e2e(args, lib, capi, tpch, stream, lineitem, n_li, world, barrier, max_over_ranks, time_e2e, AllGatherExec, q1_rows, legs):
    """Q1 from host memory through the scan boundary.  The rank's lineitem shard lies in pinned host memory as Parquet-style
    column chunks, one set per row group: sorted dictionary + bit-packed RLE_DICTIONARY pages for the low-cardinality columns
    (quantity, discount, tax, flags, ship date), PLAIN doubles for l_extendedprice (too many distinct values for a dictionary
    page, as in a real file).  Timed per step: for every row group, the encoded bytes cross PCIe (one copy per column chunk),
    sb_scan_decode rebuilds the Arrow columns in HBM, sb_hash_agg_update folds them into the aggregation state and the batch is
    released; then Final + Sort and the 4 result rows come back.  For reference the same plan is also timed from plain (decoded)
    pinned columns, 38 B/row over PCIe."""
    from spark_b200.columnar import ColumnarBatch, HostColumn, PinnedArray
    from spark_b200.execution import LocalTableScanExec
    from spark_b200.scan import decode_chunks, encode_column
    cols = tpch.Q1_COLUMNS
    ats = [lineitem.arrow_types[lineitem.column_index(c)] for c in cols]
    rg_rows = 1 << 24
    partial = tpch.q1_partial_plan(LocalTableScanExec(None), fused=True)
    # ---- untimed: write the row groups (GPU encoder) into pinned host memory ------------------------------------------------
    q1cols = lineitem.select(cols)
    groups = []
    for lo in range(0, n_li, rg_rows):
        part = q1cols.slice(lo, min(n_li, lo + rg_rows), stream)
        groups.append([encode_column(part, c, dictionary=c != "l_extendedprice", page_rows=1 << 19, stream=stream, pinned=True) for c in cols])
        part.close()
    stream.synchronize()
    enc_bytes = int(sum(ch.nbytes for g in groups for ch in g))

    from spark_b200.columnar import Stream
    copy_streams = [stream, Stream()]

    class EncodedPartial:
        """Software pipeline over the row groups: the copy + decode of row group i + 1 is queued on the other stream before the
        aggregate update of row group i waits for its own stream, so PCIe stays busy while the GPU decodes and aggregates."""

        def executeColumnar(self, stream=None):
            state = None
            nxt = decode_chunks(cols, groups[0], copy_streams[0], ats)
            try:
                for i in range(len(groups)):
                    cur, st_i = nxt, copy_streams[i % 2]
                    nxt = decode_chunks(cols, groups[i + 1], copy_streams[(i + 1) % 2], ats) if i + 1 < len(groups) else None
                    if state is None:
                        state = partial.new_state(cur)
                    state.update(cur, st_i)
                    cur.close()
                for st_i in copy_streams:
                    st_i.synchronize()
                return state.finish(stream)
            finally:
                if state is not None:
                    state.close()

    plan = tpch.q1_final_plan(AllGatherExec(EncodedPartial()), sort=True)
    capi.check(lib.sb_profile_enable(1))
    capi.check(lib.sb_profile_reset())
    ms, res = time_e2e(lambda: plan.collect(stream), max(1, args.e2e_steps))
    dms, dcnt = C.c_double(), C.c_int64()
    capi.check(lib.sb_profile_get(b"scan_decode", C.byref(dms), C.byref(dcnt)))
    capi.check(lib.sb_profile_enable(0))
    d2h = int(sum(res.column(i).nbytes for i in range(res.num_columns)))
    ok = None
    if world == 1:
        want = tpch.q1_final_plan(tpch.q1_partial_plan(LocalTableScanExec(q1cols), fused=True), sort=True).collect(stream)
        ok = check_q1(q1_rows(res), q1_rows(want))
    del groups
    # ---- the same plan from plain pinned columns (38 B/row over PCIe) ----------------------------------------------------------
    pinned = {}
    for c in cols:
        p = PinnedArray(n_li, tpch.synth_dtype(c))
        capi.check(lib.sb_table_export_host(lineitem.handle, lineitem.column_index(c), p.array.ctypes.data, None, None, None, stream.handle))
        pinned[c] = p
    stream.synchronize()
    sbt = {"l_quantity": capi.SB_FLOAT64, "l_extendedprice": capi.SB_FLOAT64, "l_discount": capi.SB_FLOAT64, "l_tax": capi.SB_FLOAT64,
           "l_returnflag": capi.SB_INT8, "l_linestatus": capi.SB_INT8, "l_shipdate": capi.SB_DATE32}
    chunk = 1 << 25

    def chunks():
        for lo in range(0, n_li, chunk):
            hi = min(n_li, lo + chunk)
            hc = [HostColumn(sbt[c], pinned[c].array[lo:hi]) for c in cols]
            yield ColumnarBatch.from_host_columns(cols, hc, stream, ats)

    class PlainPartial:
        def executeColumnar(self, stream=None):
            return partial.execute_batches(chunks(), stream)

    plain_plan = tpch.q1_final_plan(AllGatherExec(PlainPartial()), sort=True)
    pms, pres = time_e2e(lambda: plain_plan.collect(stream), 1)
    h2d_plain = int(sum(p.nbytes for p in pinned.values()))
    for p in pinned.values():
        p.close()
    q1cols.close()
    steps_run = max(1, args.e2e_steps) + 1
    return {"value": world * n_li / (ms / 1000.0), "unit": "rows/s", "ms_per_step": ms, "h2d_bytes_per_step": enc_bytes, "d2h_bytes_per_step": d2h,
            "input": "Parquet-style encoded column chunks in pinned host memory (%d-row row groups; RLE_DICTIONARY bit-packed pages, PLAIN doubles "
                     "for l_extendedprice), decoded on the GPU (sb_scan_decode) and streamed through sb_hash_agg_update" % rg_rows,
            "encoded_bytes_per_row": enc_bytes / n_li, "pcie_gbs": enc_bytes / (ms / 1000.0) / 1e9,
            "scan_decode_ms_per_step": dms.value / steps_run, "equals_resident_result": ok,
            "from_plain_columns": {"value": world * n_li / (pms / 1000.0), "ms_per_step": pms, "h2d_bytes_per_step": h2d_plain,
                                   "input": "plain pinned host columns (38 B/row), %d-row chunks streamed through sb_hash_agg_update" % chunk}}


def run_shuffle(args, lib, capi, tpch, stream, rank, world, n_orders, seed, barrier, max_over_ranks, all_true, time_resident, peak, peak_src):
    """BASELINE.json configs[3] shape: repartition(2048) of 74 B/row lineitem rows: Murmur3-pmod partition ids + stable
    multisplit on every GPU, buckets exchanged over NVLink (sb_all_to_all), no spill."""
    import torch
    import torch.distributed as dist
    from spark_b200.columnar import ColumnarBatch
    from spark_b200.execution import HashPartitioning, LocalTableScanExec, ShuffleExchangeExec
    from oracle import oracle as O
    import pyarrow as pa
    nparts = 2048
    rows = min(args.shuffle_rows, tpch.synth_rows("lineitem", n_orders))
    batch = tpch.synth_batch("lineitem", tpch.CONFIG4_COLUMNS, n_orders, seed, 0, rows, stream)
    ex = ShuffleExchangeExec(HashPartitioning(["l_orderkey"], nparts), LocalTableScanExec(batch))                  # fused: sb_shuffle_exchange
    ex2 = ShuffleExchangeExec(HashPartitioning(["l_orderkey"], nparts), LocalTableScanExec(batch), fused=False)   # sb_hash_partition + sb_all_to_all
    outs = []

    def make_step(e):
        def step():
            out = e.executeColumnar(stream)
            outs.append(out)
            while len(outs) > 1:
                outs.pop(0).close()
        return step

    steps = max(1, min(args.steps, args.leg_steps))
    names = ("partition_ids", "exchange_scatter", "partition_scatter", "a2a_transfer", "a2a_counts")
    ms2, _, prof2 = time_resident(make_step(ex2), steps, max(3, args.warmup), names)
    ms, launches, prof = time_resident(make_step(ex), steps, max(3, args.warmup), names)
    out = outs[-1]
    offs = ex.partition_offsets
    # ---- verification: (1) every received row belongs to a partition this rank owns (oracle Murmur3 on a sample), (2) rows and
    # (3) an order-independent checksum of two columns are conserved across the exchange
    lo = (rank * nparts + world - 1) // world
    hi = ((rank + 1) * nparts + world - 1) // world
    got_rows = out.num_rows
    sample = min(got_rows, 1 << 20)
    keys, _ = out.slice(0, sample, stream).column_to_numpy(0, stream) if sample else (np.zeros(0, np.int64), None)
    pid = O.partition_ids(pa.table({"l_orderkey": keys}), ["l_orderkey"], nparts) if sample else np.zeros(0, np.int32)
    ok = bool(np.all((pid >= lo) & (pid < hi))) and int(offs[-1]) == got_rows
    # the fused exchange returns the owned partitions contiguously: the sampled prefix must be sorted by partition id and agree with
    # the partition boundaries it reports
    ok = ok and bool(np.all(np.diff(pid) >= 0)) and bool(np.array_equal(pid, (np.searchsorted(offs, np.arange(sample), side="right") - 1).astype(pid.dtype)))

    def checksum(b):
        tot = []
        for name in ("l_orderkey", "l_partkey"):
            arr, _ = b.column_to_numpy(b.column_index(name), stream)
            tot.append(int(arr.sum(dtype=np.int64)))
        return tot
    before = checksum(batch)
    after = checksum(out)
    tv = torch.tensor([rows, got_rows] + before + after, dtype=torch.int64, device="cuda")
    dist.all_reduce(tv)
    tv = tv.cpu().numpy()
    ok = ok and tv[0] == tv[1] and tv[2] == tv[4] and tv[3] == tv[5]
    verified = all_true(ok)
    transport_ms = prof["exchange_scatter"][0] / steps if prof["exchange_scatter"][1] else None
    leaving = rows * tpch.CONFIG4_BYTES_PER_ROW * (world - 1) / world
    for o in outs:
        o.close()
    batch.close()
    return {"value": world * rows / (ms / 1000.0), "unit": "rows/s", "ms_per_step": ms, "steps": steps, "rows_per_gpu": rows, "num_partitions": nparts,
            "bytes_per_row": tpch.CONFIG4_BYTES_PER_ROW, "gpu_launches": int(launches), "verified": verified,
            "kernel_ms_per_step": {k: v[0] / steps for k, v in prof.items()},
            "plan": "sb_shuffle_exchange: Murmur3 pmod ids -> R-way stable multisplit whose stores land in the owners' windows over NVLink -> local split into the owned partitions",
            "variants": {"partition_then_all_to_all": {"ms_per_step": ms2, "value": world * rows / (ms2 / 1000.0),
                                                      "kernel_ms_per_step": {k: v[0] / steps for k, v in prof2.items()}}},
            "nvlink": {"bytes_leaving_each_gpu": leaving, "transport_ms": transport_ms,
                       "note": "transport = the exchange_scatter kernel: it reads every local row once and stores (R - 1) / R of them remotely",
                       "gbs_per_direction_transport_only": leaving / (transport_ms / 1000.0) / 1e9 if transport_ms else None,
                       "gbs_per_direction_whole_exchange": leaving / (ms / 1000.0) / 1e9, "peak_gbs_per_direction": 900.0},
            "roofline": {"bound": "hbm", "kernel": "hash partition (pid + multisplit)", "unit": "GB/s", "peak": peak, "peak_source": peak_src,
                         "achieved": 2 * rows * tpch.CONFIG4_BYTES_PER_ROW / (ms / 1000.0) / 1e9,
                         "frac": 2 * rows * tpch.CONFIG4_BYTES_PER_ROW / (ms / 1000.0) / 1e9 / peak,
                         "algorithmic_bytes_per_step": 2 * rows * tpch.CONFIG4_BYTES_PER_ROW, "traffic": None}}


if __name__ == "__main__":
    main()
