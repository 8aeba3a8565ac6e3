#!/usr/bin/env python
"""bench.py — rows/sec of the lineitem JOIN orders hash join + GROUP BY at SF100
per GPU (BASELINE.json metric), one process per GPU.

Workload (BASELINE.json configs[2], the configuration the metric is quoted on):

    SELECT o_orderdate, count(*), sum(l_extendedprice)
    FROM lineitem JOIN orders ON l_orderkey = o_orderkey GROUP BY o_orderdate

on synthetic TPC-H-shaped tables (include/gx_tpch_gen.h, seed 20240922).  A
"step" is one complete pass of the hot path over the datanode's resident
tables: hash build over orders, fused probe + hash aggregate over lineitem,
Finalize across datanodes (N > 1), result read back.  With N GPUs there are N
datanodes holding a SF(100*N) database placed by the reference's SHARD rule
(weak scaling; lineitem and orders are co-located on the order key, so the only
exchange is the partial-aggregate redistribute).

    python bench.py --gpus 1 --steps 10 --warmup 3
    torchrun --nproc-per-node N bench.py --gpus N ...
    python bench.py --impl reference        # the CPU executor port on the host cores
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rows/sec lineitem JOIN orders hashjoin+groupby SF100"
try:                                   # BASELINE.json names the metric; use its wording when it is there
    METRIC = json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"] or METRIC
except (OSError, ValueError, KeyError):
    pass
ALG_BYTES_PER_PROBE_ROW = 24     # SURVEY.md §8d: 8 B key + 8 B payload on hit + 8 B l_extendedprice
ALG_BYTES_PER_BUILD_ROW = 24     # 8 B key read + 16 B slot write


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ------------------------------------------------------------------ clocks
REAL_STDOUT = sys.stdout


class ClockSampler:
    """nvidia-smi clocks / throttle reasons.  The sampler needs a few hundred ms to come up
    and the timed region is short, so it is started before the warm-up steps (the GPU is under
    the same load there); stop(t0, t1) reports the samples that fall inside the timed region
    and, when the region was too short to catch any, the ones taken under load since start."""

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(prefix="clocks_", suffix=".csv")
        q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self, t0=None, t1=None):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.p:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        rows = []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(f[1]), float(f[2]), f[5:9]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except OSError:
            pass
        inside = [r for r in rows if t0 is not None and t0 <= r[0] <= t1]
        window = "timed region"
        if not inside:
            inside = [r for r in rows if t1 is None or r[0] <= t1]
            window = "warm-up + timed region (timed region shorter than the sampling period)"
        if inside:
            reasons = set()
            for r in inside:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            out = {"sm_mhz": float(np.median([r[1] for r in inside])), "sm_max_mhz": max(r[2] for r in inside),
                   "reasons": sorted(reasons), "samples": len(inside), "window": window}
        return out


# ------------------------------------------------------- CPU baseline (oracle)
def cpu_reference_run(sample_orders: int, threads: int, steps: int, warmup: int, sf: int = 100):
    """The reference CPU executor's path (oracle/: tuple-at-a-time SeqScan ->
    HashJoin -> HashAgg, the only stand-in that exists: the reference itself
    cannot be built here, SURVEY.md §8c) on `threads` host threads.  Each
    thread owns one co-partitioned slice (like one datanode / parallel worker),
    partial aggregates are combined at the end (Partial -> Finalize)."""
    import oracle as O
    import opentenbase_b200 as g
    from concurrent.futures import ThreadPoolExecutor
    bounds = np.linspace(0, sample_orders, threads + 1).astype(np.int64)
    plan = O.make_plan(outer_key_col=g.L_ORDERKEY, group_cols=[(1, 0)],
                       aggs=[(g.GX_AGG_COUNT_STAR, []), (g.GX_AGG_SUM_F8, [(g.GX_OP_COL, 1, 0)])], est_groups=2500)
    join = O.make_join(0, payload_cols=[1], inner_unique=1)

    def make(i):
        o = O.gen_orders(sf, int(bounds[i]), int(bounds[i + 1]))
        l = O.gen_lineitem(sf, int(bounds[i]), int(bounds[i + 1]))
        orel = O.Rel([O.GX_INT8, O.GX_DATE], [o[0], o[2]])
        lrel = O.Rel([O.GX_INT8, O.GX_FLOAT8], [l[0], l[2]])
        return orel, lrel, len(o[0]) + len(l[0])

    with ThreadPoolExecutor(threads) as ex:
        rels = list(ex.map(make, range(threads)))
        nrows = sum(r[2] for r in rels)

        def one(i):
            res, raw = O.exec_agg(rels[i][1], plan, rels[i][0], join, keep_raw=True)
            return raw

        times = []
        final = None
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            raws = list(ex.map(one, range(threads)))
            final = O.combine(plan, raws)
            dt = time.perf_counter() - t0
            for r in raws:
                O.lib().orc_result_free(r)
            if it >= warmup:
                times.append(dt)
    total_count = int(final.aggs[:, 0].view(np.int64).sum())
    return {"rows": nrows, "secs_per_step": float(np.mean(times)), "rows_per_sec": nrows / float(np.mean(times)),
            "count_star_total": total_count, "groups": final.ngroups, "final": final.sorted()}


def effective_cpus() -> int:
    """Host threads this process can really run at once: the affinity mask, capped by a cgroup
    CPU quota if there is one (a container may show 128 CPUs and be allowed 16 of them)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]              # cgroup v2
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())            # cgroup v1
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0 and period > 0:
                n = min(n, max(1, quota // period))
        except (OSError, ValueError):
            pass
    return max(1, n)


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    threads = effective_cpus()
    sample_orders = (args.cpu_sample_orders // 2) * threads          # ~0.75 M orders (3.75 M rows) per thread
    r = cpu_reference_run(sample_orders, threads, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["rows_per_sec"], "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["secs_per_step"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": r["rows_per_sec"], "unit": "rows/s", "cores": threads, "kind": "port",
                         "sample": f"{sample_orders} orders + their lineitem rows ({r['rows']} rows) of the SF100 tables, "
                                   f"{threads} threads, one co-partitioned slice each, partial->final combine"},
        "e2e": {"value": r["rows_per_sec"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=REAL_STDOUT, flush=True)
    return 0


def workload_config(args, world):
    return {"workload": "configs[2]: lineitem JOIN orders ON l_orderkey=o_orderkey, hash build on orders, probe lineitem, "
                        "GROUP BY o_orderdate: count(*), sum(l_extendedprice)",
            "sf_per_gpu": args.sf, "sf_total": args.sf * world, "datanodes": world,
            "parallelism": f"{world} datanode(s), one per GPU, SHARD placement on the order key",
            "l2": "inputs (>= 11 GB per GPU at SF100) are far larger than the 126 MB L2; no flush needed between steps",
            "memory": "gx_pool_reserve(0): free HBM minus 8 GB mapped into the stream-ordered pool at start-up"}


# ---------------------------------------------------------------- GPU arm
def same_result(got, want, int_aggs=(), rtol=1e-9):
    """GPU rows (keys, aggs, nulls — any order, possibly concatenated over datanodes) against a sorted
    oracle AggResult: keys and integer aggregates bit-exact, float8 aggregates within rtol relative."""
    keys, aggs, _ = got
    if keys.shape != want.keys.shape:
        return False, f"group count {keys.shape[0]} vs oracle {want.keys.shape[0]}"
    if keys.shape[0] == 0:
        return True, "0 groups"
    order = np.lexsort([keys[:, c] for c in reversed(range(keys.shape[1]))]) if keys.shape[1] else np.arange(len(keys))
    keys, aggs = keys[order], aggs[order]
    if not np.array_equal(keys, want.keys):
        return False, "group keys differ"
    for a in range(aggs.shape[1]):
        if a in int_aggs:
            if not np.array_equal(aggs[:, a].view(np.int64), want.aggs[:, a].view(np.int64)):
                return False, f"integer aggregate {a} not bit-exact"
        elif not np.allclose(aggs[:, a], want.aggs[:, a], rtol=rtol, atol=0):
            return False, f"float8 aggregate {a} beyond {rtol} relative"
    return True, f"{keys.shape[0]} groups"


def cat_results(parts):
    return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))


def dump_outputs(path, result):
    """The configs[2] answer of the last timed step (all datanodes' groups) as float64 .npy files.  The library returns
    groups in hash-table order, so rows are put in group-key order: two builds then compare array by array."""
    keys, aggs, nulls = result
    order = np.lexsort(keys.T[::-1]) if keys.shape[1] else np.arange(len(keys))
    os.makedirs(path, exist_ok=True)
    arrays = {"o_orderdate": keys[order, 0], "count_star": aggs[order, 0].view(np.int64),
              "sum_l_extendedprice": aggs[order, 1], "nulls": nulls[order]}
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def phase_table(ctx, names, steps):
    out = {}
    for name in names:
        ms, n = ctx.profile_get(name)
        if n:
            out[name] = {"ms_per_step": round(ms / steps, 4), "launches_per_step": n / steps}
    return out


PHASES = ("build_sample", "build_bounds", "build_scatter", "build", "build_clear", "build_expand", "probe_agg", "agg",
          "agg_compact", "probe_records", "scan_records", "runagg", "runagg_merge", "radix_partition", "radix_agg", "radix_overflow",
          "filter", "partition", "alltoall", "probe", "probe_count", "combine_pack", "allgather", "combine_merge",
          "combine_partition", "peer_wait_ack", "peer_scatter", "peer_publish", "peer_wait", "peer_gather", "peer_ack")


def run_ours(args):
    import opentenbase_b200 as g
    from opentenbase_b200 import plans as P
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", ""):
        os.environ["NCCL_DEBUG"] = "WARN"          # NCCL prints its version banner to stdout otherwise
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = g.Context(local_rank)
    if world > 1:
        box = [g.Context.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        ctx.comm_init(rank, world, box[0])
    ctx.set_shardmap(world)
    ctx.pool_reserve(0)         # map the HBM the queries will use into the stream-ordered pool once, not mid-query

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()

    def allred(x, op):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def allmax(x):
        return allred(x, dist.ReduceOp.MAX if dist else None)

    def allsum(x):
        return allred(x, dist.ReduceOp.SUM if dist else None)

    def gather0(obj):
        if dist is None:
            return [obj]
        box = [None] * world if rank == 0 else None
        dist.gather_object(obj, box, dst=0)
        return box

    sf_total = args.sf * world
    n_orders_total = 1_500_000 * sf_total
    n_cust_total = 150_000 * sf_total
    cap_o = int(1_500_000 * args.sf * 1.03) + 1_000_000
    cap_l = int(6_000_000 * args.sf * 1.03) + 4_000_000
    cap_c = int(150_000 * args.sf * 1.05) + 100_000
    # full schemas: config 3 reads (orderkey, orderdate) x (orderkey, extendedprice); Q1 and Q3 read the rest
    ot = ctx.table(g.SCHEMAS[g.T_ORDERS], cap_o).generate(g.T_ORDERS, sf_total, 0, n_orders_total, rank, world)
    lt = ctx.table(g.SCHEMAS[g.T_LINEITEM], cap_l).generate(g.T_LINEITEM, sf_total, 0, n_orders_total, rank, world)
    ct = ctx.table(g.SCHEMAS[g.T_CUSTOMER], cap_c).generate(g.T_CUSTOMER, sf_total, 0, n_cust_total, rank, world)
    no, nl, nc = ot.nrows, lt.nrows, ct.nrows
    plan = P.config3_plan(g.L_ORDERKEY, g.L_EXTENDEDPRICE)

    def step(o=ot, l=lt):
        ht = ctx.hash_build(o, g.O_ORDERKEY, [g.O_ORDERDATE], unique=True)
        r = ctx.hash_agg(l, plan, ht)
        r.combine()
        out = r.fetch()
        r.free(); ht.free()
        return out

    clocks = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(args.warmup):
        step()
    # ---- timed region: exactly K steps, device events on the library's stream
    ctx.profile(True)
    launches0 = ctx.launches
    barrier()
    t0 = time.perf_counter(); wall0 = time.time()
    ctx.timer_start()
    last = None
    for _ in range(args.steps):
        last = step()
    dev_ms = ctx.timer_stop()
    ctx.sync()
    wall_ms = (time.perf_counter() - t0) * 1e3; wall1 = time.time()
    barrier()
    launches = ctx.launches - launches0
    clk = clocks.stop(wall0, wall1) if clocks else None
    probe_ms, probe_n = ctx.profile_get("probe_agg")
    _, seg_n = ctx.profile_get("probe_agg_seg")          # > 0: the streamed-table variant (gx_k_runjoin_seg) ran
    _, tma_n = ctx.profile_get("probe_agg_tma")          # > 0: the rows-by-copy-engine variant (gx_k_runjoin_tma) ran
    build_ms, build_n = ctx.profile_get("build")
    phases = phase_table(ctx, PHASES, args.steps)
    ctx.profile(False)
    dev_ms_max = allmax(dev_ms)
    wall_ms_max = allmax(wall_ms)
    rows_all = allsum(float(no + nl))
    ms_per_step = dev_ms_max / args.steps
    value = rows_all / (ms_per_step / 1e3)
    # size-independent correctness properties on the last step's result
    keys, aggs, nulls = last
    count_local = int(aggs[:, 0].view(np.int64).sum())
    count_total = allsum(float(count_local))
    nl_total = allsum(float(nl))
    checks = {"count_star_equals_lineitem_rows": int(count_total) == int(nl_total),
              "groups_this_node": int(len(keys))}
    if args.dump_outputs:
        parts = gather0(last)
        if rank == 0:
            dump_outputs(args.dump_outputs, cat_results(parts))

    # ---- the other BASELINE configurations, same run, same tables (extras; the headline stays configs[2])
    extras = {}
    cols = {"c": {"custkey": g.C_CUSTKEY, "mktsegment": g.C_MKTSEGMENT},
            "o": {"orderkey": g.O_ORDERKEY, "custkey": g.O_CUSTKEY, "orderdate": g.O_ORDERDATE, "shippriority": g.O_SHIPPRIORITY},
            "l": {"orderkey": g.L_ORDERKEY, "extendedprice": g.L_EXTENDEDPRICE, "discount": g.L_DISCOUNT, "shipdate": g.L_SHIPDATE}}
    q1plan = P.q1_plan(g.L_QUANTITY, g.L_EXTENDEDPRICE, g.L_DISCOUNT, g.L_TAX, g.L_SHIPDATE, g.L_RETURNFLAG, g.L_LINESTATUS)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

    def timed_block(fn, steps, warm=2):
        for _ in range(warm):
            fn()
        ctx.profile(True)
        l0 = ctx.launches
        barrier()
        ctx.timer_start()
        for _ in range(steps):
            out = fn()
        ms = ctx.timer_stop()
        ctx.sync()
        barrier()
        ph = phase_table(ctx, PHASES, steps)
        ctx.profile(False)
        return allmax(ms) / steps, ph, out, (ctx.launches - l0) // steps

    xsteps = max(1, min(args.steps, args.extra_steps))
    if not args.no_extras:
        # Q3 shape (configs[3]/[4]): two NCCL redistributes per step
        q3stats = {}

        def q3():
            r = P.q3_datanode(ctx, ct, ot, lt, cols["c"], cols["o"], cols["l"], q3stats)
            out = r.fetch(pinned=True)            # a million groups: the result lands in reusable pinned buffers
            r.free()
            return out
        ms, ph, out, nlaunch = timed_block(q3, xsteps)
        rows3 = allsum(float(nc + no + nl))
        sent = allsum(float(q3stats["bytes_sent"]))
        builds = allsum(float(q3stats["cust_kept"] + q3stats["build_rows"]))
        alg = 28.0 * allsum(float(nl)) + 20.0 * allsum(float(no)) + 5.0 * allsum(float(nc)) + 16.0 * builds + 2.0 * sent
        a2a_ms = ph.get("alltoall", {}).get("ms_per_step", 0.0)
        peer_ms = sum(ph.get(k, {}).get("ms_per_step", 0.0) for k in ("peer_scatter", "peer_publish", "peer_wait"))
        transport = "nccl send/recv after a local partition"
        if peer_ms and not a2a_ms:
            # rows were stored straight into the destinations' windows by the routing kernel: the exchange is that kernel
            # plus the wait for the slowest peer's rows
            a2a_ms, transport = peer_ms, "peer windows: the routing kernel stores into the destination's HBM over NVLink (no partition, no collective)"
        extras["q3"] = {"workload": "configs[3] shape: customer JOIN orders JOIN lineitem, Distribute by o_custkey, then by o_orderkey; "
                                    "sum(l_extendedprice*(1-l_discount)) GROUP BY l_orderkey, o_orderdate, o_shippriority",
                        "ms_per_step": ms, "rows_per_s": rows3 / (ms / 1e3), "rows_per_step": rows3, "steps": xsteps,
                        "groups_total": allsum(float(len(out[0]))), "launches_per_step": nlaunch,
                        "redistributed_rows": allsum(float(q3stats["redistributed_custkey"] + q3stats["redistributed_orderkey"])),
                        "alltoall_bytes_per_gpu": sent / world, "alltoall_ms": a2a_ms, "transport": transport if world > 1 else None,
                        "nvlink_gb_s_per_gpu": (sent / world * (world - 1) / world / (a2a_ms / 1e3) / 1e9) if (a2a_ms and world > 1) else None,
                        "nvlink_peak_gb_s": 900.0,
                        "algorithmic_bytes": alg, "hbm_gb_s_per_gpu": alg / world / (ms / 1e3) / 1e9,
                        "frac_hbm": alg / world / (ms / 1e3) / 1e9 / peak, "phases_ms": ph,
                        "host_ms_per_call_last_step": {k: round(v, 3) for k, v in q3stats.get("host_ms_per_call", {}).items()}}

        # Q1 shape (configs[4]): Partial HashAggregate -> all-gather of partial states -> Finalize
        def q1():
            r = ctx.hash_agg(lt, q1plan)
            r.combine()
            out = r.fetch()
            r.free()
            return out
        ms, ph, out, nlaunch = timed_block(q1, xsteps)
        rows1 = allsum(float(nl))
        q1count = allsum(float(out[1][:, 7].view(np.int64).sum()))
        extras["q1"] = {"workload": "configs[4] Q1 shape: 8 aggregates GROUP BY l_returnflag, l_linestatus, l_shipdate qual, partial->final across datanodes",
                        "ms_per_step": ms, "rows_per_s": rows1 / (ms / 1e3), "steps": xsteps, "groups_total": allsum(float(len(out[0]))),
                        "launches_per_step": nlaunch, "algorithmic_bytes": 38.0 * rows1,
                        "hbm_gb_s_per_gpu": 38.0 * rows1 / world / (ms / 1e3) / 1e9, "frac_hbm": 38.0 * rows1 / world / (ms / 1e3) / 1e9 / peak,
                        "count_star_total": q1count, "phases_ms": ph}
        # configs[0] and configs[1] shapes on the GPU (kernel-level; configs[0] itself is the CPU-only case)
        for name, pl, bpr in (("config1", P.config1_plan(g.L_RETURNFLAG), 1.0), ("config2", P.config2_plan(g.L_SHIPDATE, g.L_EXTENDEDPRICE), 12.0)):
            def cfg(pl=pl):
                r = ctx.hash_agg(lt, pl)
                r.combine()
                out = r.fetch()
                r.free()
                return out
            ms, ph, out, nlaunch = timed_block(cfg, xsteps)
            extras[name] = {"ms_per_step": ms, "rows_per_s": rows1 / (ms / 1e3), "groups_total": allsum(float(len(out[0]))),
                            "frac_hbm": bpr * rows1 / world / (ms / 1e3) / 1e9 / peak, "phases_ms": ph}

    # ---- the same configs[2] query over UNCLUSTERED copies of both tables (rows permuted): neither the key-ordered
    # build nor the run-folding probe applies; every probe is a random 32-byte sector of a table far larger than L2
    if not args.no_extras and not args.no_unclustered:
        lp = ctx.scan_filter(lt, [], [g.L_ORDERKEY, g.L_EXTENDEDPRICE]); lu = lp.permuted(7); lp.free()
        op_ = ctx.scan_filter(ot, [], [g.O_ORDERKEY, g.O_ORDERDATE]); ou = op_.permuted(11); op_.free()
        uplan = P.config3_plan(0, 1)

        def ustep():
            ht = ctx.hash_build(ou, 0, [1], unique=True)
            r = ctx.hash_agg(lu, uplan, ht)
            r.combine()
            out = r.fetch()
            r.free(); ht.free()
            return out
        ms, ph, out, nlaunch = timed_block(ustep, xsteps, warm=1)
        ucount = allsum(float(out[1][:, 0].view(np.int64).sum()))
        pm = ph.get("probe_agg", {}).get("ms_per_step")
        extras["unclustered"] = {"workload": "configs[2] query, both tables row-permuted (out[i] = in[(i*A+B) mod n])",
                                 "ms_per_step": ms, "value_unclustered": rows_all / (ms / 1e3), "launches_per_step": nlaunch,
                                 "count_star_equals_lineitem_rows": int(ucount) == int(nl_total),
                                 "probe_sectors_gb_s": (nl * 32.0 / (pm / 1e3) / 1e9) if pm else None,
                                 "probe_alg_frac_hbm": (nl * 24.0 / (pm / 1e3) / 1e9 / peak) if pm else None,
                                 "note": "one 32-byte DRAM sector per probe is the floor for an unpartitioned probe of a table larger than L2 "
                                         "(B200 delivers ~42 G random gathers/s, profiles/r01_ubench_random_access.txt)",
                                 "phases_ms": ph}
        checks["unclustered_count_star_equals_lineitem_rows"] = extras["unclustered"]["count_star_equals_lineitem_rows"]
        lu.free(); ou.free()

    # ---- parity against the oracle on a slice, through the same calls (all datanodes take part)
    nslice = min(args.cpu_sample_orders, n_orders_total)
    os_ = ctx.table(g.SCHEMAS[g.T_ORDERS], nslice + 1024).generate(g.T_ORDERS, sf_total, 0, nslice, rank, world)
    ls_ = ctx.table(g.SCHEMAS[g.T_LINEITEM], nslice * 7 + 1024).generate(g.T_LINEITEM, sf_total, 0, nslice, rank, world)
    got3 = step(os_, ls_)
    gotq1 = gotq3 = None
    if not args.no_extras:
        r = ctx.hash_agg(ls_, q1plan); r.combine(); gotq1 = r.fetch(); r.free()
        r = P.q3_datanode(ctx, ct, os_, ls_, cols["c"], cols["o"], cols["l"]); gotq3 = r.fetch(); r.free()
    gathered = gather0((got3, gotq1, gotq3))
    os_.free(); ls_.free()

    # ---- end to end: HOST (pinned) buffers -> result, copies inside the timed region
    e2e = None
    try:
        e2e = run_e2e(ctx, g, ot, lt, no, nl, plan, args, barrier, allmax, rows_all)
    except g.GxError as ex:
        e2e = {"value": None, "unit": "rows/s", "error": str(ex)}

    e2e_pages = None
    if rank == 0 and not args.no_extras and args.pages_gb > 0:
        try:
            e2e_pages = run_e2e_pages(ctx, g, args)
        except Exception as ex:                                  # an extra must never take the headline line down with it
            e2e_pages = {"error": repr(ex)}

    fnpage = None
    if rank == 0 and not args.no_extras:
        try:
            fnpage = run_fnpage(ctx, g, ot, cols["o"], peak)
        except Exception as ex:
            fnpage = {"error": repr(ex)}

    if rank != 0:
        ctx.close()
        if dist is not None:
            dist.destroy_process_group()
        return 0

    probe_avg_ms = probe_ms / max(probe_n, 1)
    achieved = nl * ALG_BYTES_PER_PROBE_ROW / (probe_avg_ms / 1e3) / 1e9 if probe_n else None
    traffic = None
    traffic_src = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "probe_agg_traffic.json")))
        if seg_n or tma_n:
            tj = tj.get("gx_k_runjoin_seg" if seg_n else "gx_k_runjoin_tma") or {}
        traffic = tj.get("dram_bytes_per_launch_sf100")
        if traffic:
            traffic_src = "profiles/probe_agg_traffic.json (ncu --set full capture of this kernel at SF100, " + str(tj.get("source", "")) + "); not measured in this run"
    except (OSError, ValueError):
        pass
    probe_kernel = ("gx_k_runjoin_seg (fused hash probe + hash aggregate over lineitem; join table streamed through a cp.async.bulk/mbarrier ring)"
                    if seg_n else
                    "gx_k_runjoin_tma (fused hash probe + hash aggregate over lineitem; outer rows delivered by cp.async.bulk onto per-warp mbarriers)"
                    if tma_n else "gx_k_runjoin (fused hash probe + hash aggregate over lineitem)")
    roofline = {"kernel": probe_kernel, "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                "traffic": traffic, "traffic_source": traffic_src,
                "frac_dram": (traffic * (nl / 600_000_105.0) / (probe_avg_ms / 1e3) / 1e9 / peak) if (traffic and probe_n) else None,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": nl * ALG_BYTES_PER_PROBE_ROW, "avg_launch_ms": probe_avg_ms,
                "note": "achieved/frac use SURVEY 8d's 24 B per probe row; frac_dram uses the DRAM bytes ncu measured for this kernel "
                        "(compact 8-byte slots move fewer bytes than 8d charges), scaled to this run's row count",
                "build_kernel_avg_ms": build_ms / max(build_n, 1),
                "build_alg_GBps": (no * ALG_BYTES_PER_BUILD_ROW / (build_ms / max(build_n, 1) / 1e3) / 1e9) if build_n else None}

    # ---- CPU baseline (oracle, 1 thread) on the parity slice; its result IS the parity reference for configs[2]
    import oracle as O
    r = cpu_reference_run(nslice, 1, 1, 0, sf_total)
    cpu = {"value": r["rows_per_sec"], "unit": "rows/s", "cores": 1, "kind": "port",
           "sample": f"first {nslice} orders and their lineitem rows ({r['rows']} rows) of the SF{sf_total} tables (an SF{sf_total} SLICE: "
                     "its hash table is ~100 MB, friendlier to the CPU than the full build side), "
                     "oracle/ tuple-at-a-time executor, 1 thread (one backend per datanode fragment)"}
    ok, why = same_result(cat_results([x[0] for x in gathered]), r["final"], int_aggs=(0,))
    checks["config3_parity_vs_oracle"] = ok
    checks["config3_parity_detail"] = f"{why}; slice of {nslice} orders over {world} datanode(s); count(*) bit-exact, sum within 1e-9"
    if not args.no_extras:
        l = O.gen_lineitem(sf_total, 0, nslice)
        want = O.exec_agg(O.Rel(g.SCHEMAS[g.T_LINEITEM], l),
                          P.q1_plan(g.L_QUANTITY, g.L_EXTENDEDPRICE, g.L_DISCOUNT, g.L_TAX, g.L_SHIPDATE, g.L_RETURNFLAG, g.L_LINESTATUS,
                                    maker=O.make_plan)).sorted()
        ok, why = same_result(cat_results([x[1] for x in gathered]), want, int_aggs=(7,))
        checks["q1_parity_vs_oracle"] = ok; checks["q1_parity_detail"] = why
        want = O.q3_reference(sf_total, nslice, n_cust_total, P.DATE_Q3, P.SEGMENT_Q3)
        ok, why = same_result(cat_results([x[2] for x in gathered]), want)
        checks["q3_parity_vs_oracle"] = ok; checks["q3_parity_detail"] = why
    failed = [k for k, v in checks.items() if v is False]

    line = {"metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "wall_ms_per_step": wall_ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
            "config": workload_config(args, world), "rows_per_step": rows_all,
            "e2e": e2e, "gpu_launches": launches, "clocks": clk, "roofline": roofline, "cpu_baseline": cpu, "checks": checks,
            "float_determinism": "float8 sums use shared-memory atomics: not bit-identical run to run, within 1e-9 relative of the reference",
            "phases_ms": phases}
    line.update(extras)
    if e2e_pages is not None:
        line["e2e_pages"] = e2e_pages
        if e2e_pages.get("rows_match_oracle") is False:
            failed.append("e2e_pages.rows_match_oracle")
    if fnpage is not None:
        line["fnpage"] = fnpage
        if fnpage.get("round_trip_equal") is False:
            failed.append("fnpage.round_trip_equal")
    print(json.dumps(line), file=REAL_STDOUT, flush=True)
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    if failed:
        print(f"bench: FAILED checks: {failed}", file=sys.stderr)
        return 1
    return 0


def run_e2e(ctx, g, ot, lt, no, nl, plan, args, barrier, allmax, rows_all):
    """configs[2] through gx_exec_host(): HOST column buffers in, finalized HOST result out, every step."""
    from opentenbase_b200 import plans as P
    sizes = [(ot, g.O_ORDERKEY, 8, no), (ot, g.O_ORDERDATE, 4, no), (lt, g.L_ORDERKEY, 8, nl), (lt, g.L_EXTENDEDPRICE, 8, nl)]
    bufs = []
    for t, col, sz, n in sizes:
        p = ctx.host_alloc(max(n * sz, 8))
        ctx._chk(g.lib().gx_table_read_column(t.h, col, 0, n, p, None))     # fill the pinned staging buffer
        bufs.append(p)
    h2d = sum(sz * n for _, _, sz, n in sizes)
    steps = max(1, min(args.steps, args.e2e_steps))
    hplan = P.config3_plan(0, 1)                 # host tables carry only the referenced columns

    def estep():
        r = ctx.exec_host([g.GX_INT8, g.GX_FLOAT8], bufs[2:4], nl, hplan, [g.GX_INT8, g.GX_DATE], bufs[0:2], no,
                          inner_key_col=0, payload_cols=[1], inner_unique=True)
        r.combine()
        out = r.fetch()
        r.free()
        return out

    # what the link can do from this very staging memory, same run: one stream and four streams
    ceiling1 = ctx.h2d_probe(bufs[2], min(nl * 8, 2 << 30), 1)
    ceiling4 = ctx.h2d_probe(bufs[2], min(nl * 8, 2 << 30), 4)
    estep()                                   # warm-up
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = estep()
    ctx.sync()
    dt = time.perf_counter() - t0
    barrier()
    dt = allmax(dt)
    d2h = int(out[0].nbytes + out[1].nbytes + out[2].nbytes)
    placement = staging_placement(bufs)
    for p in bufs:
        ctx.host_free(p)
    rate = h2d / (dt / steps) / 1e9
    ceiling = max(ceiling1, ceiling4)
    return {"value": rows_all / (dt / steps), "unit": "rows/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": d2h,
            "steps": steps, "ms_per_step": dt / steps * 1e3, "h2d_gb_per_s": rate,
            "pcie_ceiling_gb_s": ceiling, "pcie_ceiling_1_stream_gb_s": ceiling1, "pcie_ceiling_4_streams_gb_s": ceiling4,
            "frac_of_pcie_ceiling": rate / ceiling if ceiling else None, "staging": placement,
            "note": "gx_exec_host: pinned host columns -> HBM (chunked over the copy streams, the build overlaps the outer upload) -> "
                    "build -> probe+agg -> result on the host, every step; pcie_ceiling = cudaMemcpyAsync of 2 GB from the same "
                    "staging buffer in the same run"}


def run_fnpage(ctx, g, ot, ocols, peak, rows=20_000_000):
    """The reference's redistribute wire format on the device: `rows` orders rows (orderkey, custkey, orderdate, shippriority -
    the tuple of Q3's first Distribute) -> FnPages -> rows.  Kernel times from the library's launch profile; the calls also
    move the pages over PCIe (pageable host memory here), which is not the kernels' business."""
    keep = [ocols["orderkey"], ocols["custkey"], ocols["orderdate"], ocols["shippriority"]]
    # TPC-H order keys use 8 of every 32 values: key <= 4 * rows keeps about `rows` rows (of this datanode's share)
    t = ctx.scan_filter(ot, [(ocols["orderkey"], g.GX_LE, 4 * rows)], keep)
    sizes = {g.GX_INT8: (8, 8), g.GX_INT4: (4, 4), g.GX_DATE: (4, 4), g.GX_FLOAT8: (8, 8), g.GX_CHAR: (1, 1)}
    al, ag = [sizes[x][0] for x in t.types], [sizes[x][1] for x in t.types]
    for it in range(2):                                 # the first pass loads the kernels (lazy module loading) and is not reported
        ctx.profile(True)
        pages = ctx.fnpage_pack(t, al, ag, g.GxFnPageId(1, 1, 1, 0, 0, 0, 0), True)
        pack_ms, _ = ctx.profile_get("fnpage_pack")
        ctx.profile(False); ctx.profile(True)
        back = ctx.fnpage_unpack(pages, al, ag, list(range(len(al))), list(t.types), notnull=[1] * len(al))
        unpack_ms, _ = ctx.profile_get("fnpage_unpack")
        ctx.profile(False)
        if it == 0:
            back.free()
    ok = back.nrows == t.nrows and all(np.array_equal(back.read(c), t.read(c)) for c in range(len(al)))
    row_bytes = sum(al)
    out = {"workload": "orders rows of Q3's first Distribute as FnPages (forward/fnbufpage.h): columns -> pages -> columns",
           "rows": int(t.nrows), "pages": int(len(pages)), "tuple_bytes_on_the_wire": int(pages[0, 32:36].copy().view(np.uint32)[0]),
           "pack_kernel_ms": pack_ms, "unpack_kernels_ms": unpack_ms, "round_trip_equal": bool(ok),
           # sender: read the columns, write the pages (+ the memset that defines every byte); receiver: read the pages twice (count, deform), write the columns
           "pack_gb_s": (t.nrows * row_bytes + 2 * len(pages) * 8192) / (pack_ms / 1e3) / 1e9 if pack_ms else None,
           "unpack_gb_s": (t.nrows * row_bytes + 2 * len(pages) * 8192) / (unpack_ms / 1e3) / 1e9 if unpack_ms else None,
           "hbm_peak_gb_s": peak}
    back.free(); t.free()
    return out


def run_e2e_pages(ctx, g, args):
    """The plug-in's real ingest path at scale: raw 8 KB heap pages (built by the oracle's page writer, TPC-H lineitem
    layout, 8 attributes) + heapgetpage()-style visibility lists -> gx_stage_acquire ring -> gx_table_append_heap_pages ->
    device deform of the 4 referenced attributes, 32 MB batches, no synchronisation per batch.  The page set (~0.5 GB)
    is replayed until `--pages-gb` GB have gone through, like a relation that many pages long."""
    import ctypes as C
    import oracle as O
    nord = 1_250_000
    l = O.gen_lineitem(100, 0, nord)
    ltypes = [O.GX_INT8, O.GX_FLOAT8, O.GX_FLOAT8, O.GX_FLOAT8, O.GX_FLOAT8, O.GX_DATE, O.GX_CHAR, O.GX_CHAR]
    rel = O.Rel(ltypes, l)
    pages = rel.pages()
    npages, ntup = rel.npages, rel.ntuples
    L = O.lib()
    L.orc_heapgetpage.restype = C.c_int
    L.orc_heapgetpage.argtypes = [C.c_void_p, C.c_void_p]
    stride = 291                                                  # MaxHeapTuplesPerPage
    vis = np.zeros((npages, stride), np.uint16); cnt = np.zeros(npages, np.int32)
    for p in range(npages):
        cnt[p] = L.orc_heapgetpage(pages[p * 8192:].ctypes.data, vis[p].ctypes.data)
    reps = max(1, int(round(args.pages_gb * 1e9 / (npages * 8192.0))))
    attnums = [0, 2, 3, 5]                                        # l_orderkey, l_extendedprice, l_discount, l_shipdate
    d = g.GxHeapDesc()
    d.natts, d.ncols = 8, 4
    for i, (ln, al) in enumerate(zip([8, 8, 8, 8, 8, 4, 1, 1], [8, 8, 8, 8, 8, 4, 1, 1])):
        d.att_len[i], d.att_align[i], d.att_notnull[i] = ln, al, 1
    for i, a in enumerate(attnums):
        d.attnums[i] = a
    t = ctx.table([g.GX_INT8, g.GX_FLOAT8, g.GX_FLOAT8, g.GX_DATE], int(ntup * reps * 1.01) + 1024)
    B = 4096
    pb, vb = B * 8192, B * stride * 2
    slot_bytes = pb + vb + B * 4

    def load():
        t.truncate()
        for _ in range(reps):
            for p0 in range(0, npages, B):
                n = min(B, npages - p0)
                slot = ctx.stage_acquire(slot_bytes)
                C.memmove(slot, pages[p0 * 8192:].ctypes.data, n * 8192)               # the provider's memcpy out of shared_buffers
                C.memmove(slot + pb, vis[p0].ctypes.data, n * stride * 2)
                C.memmove(slot + pb + vb, cnt[p0:].ctypes.data, n * 4)
                ctx._chk(g.lib().gx_table_append_heap_pages(t.h, slot, n, C.byref(d), slot + pb, slot + pb + vb, stride))
        ctx._chk(g.lib().gx_table_load_finish(t.h))
    load()                                                        # warm-up (pins the ring, grows nothing afterwards)
    t0 = time.perf_counter()
    load()
    dt = time.perf_counter() - t0
    # host-side copy rate alone (what heapgetpage + memcpy can feed at best from one backend process)
    slot = ctx.stage_acquire(slot_bytes)
    t1 = time.perf_counter()
    for p0 in range(0, npages, B):
        C.memmove(slot, pages[p0 * 8192:].ctypes.data, min(B, npages - p0) * 8192)
    host_gbs = npages * 8192 / (time.perf_counter() - t1) / 1e9
    ok = t.nrows == ntup * reps
    first = np.empty(ntup, np.int64)
    ctx._chk(g.lib().gx_table_read_column(t.h, 0, 0, ntup, first.ctypes.data, None))
    ok = ok and bool(np.array_equal(first, l[0]))
    t.free()
    gb = npages * 8192.0 * reps / 1e9
    return {"page_gb": gb, "rows": int(ntup * reps), "seconds": dt, "page_gb_per_s": gb / dt, "rows_per_s": ntup * reps / dt,
            "host_memcpy_gb_per_s": host_gbs, "rows_match_oracle": ok,
            "note": "one host thread copies every page into the pinned ring (as gpuexec_load_relation does out of shared_buffers) while the "
                    "previous batch's DMA and deform run; the ceiling of this leg is that single-thread memcpy, not PCIe"}


def staging_placement(bufs):
    """Where the pinned staging buffers ended up (pages per NUMA node, from /proc/self/numa_maps) and the
    node the GPU hangs off: the e2e figure halves when the two differ (DESIGN.md §5)."""
    info = {}
    try:
        want = {int(p) for p in bufs}
        pages = {}
        for line in open("/proc/self/numa_maps"):
            f = line.split()
            if int(f[0], 16) in want:
                for tok in f[1:]:
                    if tok[0] == "N" and "=" in tok:
                        node, n = tok[1:].split("=")
                        pages[node] = pages.get(node, 0) + int(n)
        info["pages_by_node"] = pages
    except (OSError, ValueError, IndexError):
        pass
    try:
        bus = subprocess.check_output(["nvidia-smi", f"--id={env_int('LOCAL_RANK', 0)}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                      text=True, stderr=subprocess.DEVNULL).strip().lower()
        bus = bus[-12:] if len(bus) > 12 else bus                     # 00000000:1B:00.0 -> 0000:1b:00.0
        info["gpu_numa_node"] = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
    except (OSError, ValueError, subprocess.SubprocessError):
        pass
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sf", type=int, default=100, help="scale factor per GPU")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--extra-steps", type=int, default=5, help="timed steps of the Q3/Q1/config1/config2 extras")
    ap.add_argument("--no-extras", action="store_true", help="headline only (profiling runs)")
    ap.add_argument("--no-unclustered", action="store_true", help="skip the row-permuted variant")
    ap.add_argument("--pages-gb", type=float, default=10.0, help="GB of heap pages pushed through the page loader (e2e_pages leg; 0 = skip)")
    ap.add_argument("--cpu-sample-orders", type=int, default=1_500_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline query's answer from the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    # stdout carries exactly one JSON line: anything a library prints on fd 1 meanwhile (NCCL's
    # version banner, for one) is sent to stderr instead
    global REAL_STDOUT
    sys.stdout.flush()
    REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
