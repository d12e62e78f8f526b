#!/usr/bin/env python
"""bench.py -- the north-star measurement: rows/s for select -> fetch -> sum/min/max over
the 4 B-row int32 table of BASELINE.json config 5, row-range partitioned into 8 shards of
500 M rows (positions are int32, /root/reference/src/query.c:94-95, so a shard must stay
below 2^31 rows) spread over N B200s, aggregate partials combined with an NCCL allreduce.

One "step" = one pass of the chain over every shard of the table on every rank:
  s = select(tbl.col1, lo, hi)      (query.c:92)    } adb_chain_select_fetch_agg: two kernels per
  f = fetch(tbl.col2, s)            (query.c:223)   } shard -- the predicate pass (mask_kernel), then
  a = sum(f) / min(f) / max(f)      (query.c:325..) } the expansion with gather + aggregates fused in
with the position list and the fetched vector still materialised, as the operator API defines
(`value`, device-timed).  `e2e` is the same chain through the reference's own operator API
(select_column -> fetch_column -> sum of include/adb_query_api.h) from ONE host process that
drives all N GPUs (host/query_shim.c), wall clock, every count and sum read back by the host.

  python bench.py [--gpus N] [--steps K] [--warmup W]            engine arm
  python bench.py ... --dump-outputs DIR                          + what the last timed step computed
  python bench.py --impl reference ...                           reference CPU arm
N > 1 is launched by torchrun (one rank per GPU); total work is fixed (strong scaling).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TOTAL_ROWS = 4_000_000_000
N_SHARDS = 8
SEED = 42
SPAN = 1 << 30                       # col1 uniform in [0, 2^30)
FETCH_LO, FETCH_SPAN = 2**31 - 10000, 10000     # col2 near INT_MAX (milestone1.py:119)
NOMINAL_GBS = 8000.0                # the ~8 TB/s per-GPU figure north_star quotes
# the e2e leg drives the table as 2 columns of 2 B rows (a reference column holds < 2^31 rows:
# positions are int, src/query.c:94-95), each row-range sharded over the N GPUs by the shim
E2E_PARTS, E2E_PART_ROWS = 2, 2_000_000_000
DUMP_SAMPLE = 1 << 18                # list entries per shard that --dump-outputs keeps
METRIC = "rows/sec for select+fetch+sum"
UNIT = "rows/s"


def predicate(selectivity: float):
    lo = 1000
    return lo, lo + int(SPAN * selectivity)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region, in-process through NVML
    (a sample every ~2 ms; the timed region is tens of milliseconds, too short for an
    `nvidia-smi -lms` child to report from).  Falls back to one nvidia-smi query."""
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
            "sw_power_cap": 0x4}

    def __init__(self, index: int):
        self.index, self.sm, self.reasons, self.max_mhz = index, [], 0, None
        self._stop = threading.Event()
        self._thread = None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
        try:
            self.reasons |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            try:
                self.reasons |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:
                pass

    def _loop(self):
        while not self._stop.is_set():
            self._sample()
            time.sleep(0.002)

    def start(self):
        if self.nvml is None:
            return
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self._thread.join()
            if not self.sm:
                self._sample()
            return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(k for k, b in self.BITS.items() if self.reasons & b),
                    "samples": len(self.sm), "source": "nvml, sampled inside the timed region"}
        try:
            out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm",
                                  "--format=csv,noheader,nounits", "-i", str(self.index)],
                                 stdout=subprocess.PIPE, text=True, timeout=10).stdout.split(",")
            return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "reasons": [],
                    "samples": 1, "source": "nvidia-smi after the timed region (NVML unavailable)"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}


# ------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU operators on the host cores
# ------------------------------------------------------------------------------------------
def host_columns(rows: int, first_row: int, threads: int):
    """The same rows the GPU scans, regenerated on the host (counter-based generator)."""
    from analytical_database_b200 import synth
    from concurrent.futures import ThreadPoolExecutor
    sel = np.empty(rows, np.int32)
    fet = np.empty(rows, np.int32)
    chunk = 1 << 24

    def fill(b):
        e = min(rows, b + chunk)
        sel[b:e] = synth.uniform(e - b, SEED, first_row + b, 0, SPAN)
        fet[b:e] = synth.uniform(e - b, SEED + 1, first_row + b, FETCH_LO, FETCH_SPAN)

    with ThreadPoolExecutor(max(1, threads)) as ex:
        list(ex.map(fill, range(0, rows, chunk)))
    return sel, fet


def cpu_ops():
    from oracle import oracle
    ref = oracle.reference("O2")
    if ref is not None:
        return ref, "reference", "oracle/_ref/libref_O2.so = unmodified reference query.c at -O2"
    return oracle.port(), "port", "oracle/liboracle.so restatement at -O2"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    ops, kind, what = cpu_ops()
    lo, hi = predicate(args.selectivity)
    from oracle import oracle
    # the whole table, shard by shard (a reference column holds < 2^31 rows: int positions),
    # regenerated on the host outside the timed region; fewer shards only if RAM is short
    shard_rows = TOTAL_ROWS // N_SHARDS
    shards = N_SHARDS if args.cpu_rows <= 0 else max(1, min(N_SHARDS, args.cpu_rows // shard_rows))
    try:
        avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
        shards = max(1, min(shards, int(avail * 0.6) // (8 * shard_rows)))
    except (ValueError, OSError):
        pass
    cols = []
    for k in range(shards):
        cols.append((oracle.synth_uniform(shard_rows, SEED, k * shard_rows, 0, SPAN, cores),
                     oracle.synth_uniform(shard_rows, SEED + 1, k * shard_rows, FETCH_LO, FETCH_SPAN, cores)))
    rows = shard_rows * shards

    def step():
        tot = hits = 0
        for sel, fet in cols:
            a, b = ops.chain_select_fetch_sum(sel, fet, lo, hi, threads=cores)
            tot += a
            hits += b
        return tot, hits
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        s, h = step()
    dt = time.perf_counter() - t0
    value = rows * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int32 (int64 accumulate)", "data": "synthetic",
        "config": workload_config(args, rows_per_step=rows),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{shards} of the table's {N_SHARDS} shards ({rows} rows) per step, one "
                                   f"reference instance per row range on {cores} threads; {what}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "check": {"sum": s, "hits": h},
    }
    emit(line)
    return 0


def workload_config(args, rows_per_step):
    return {
        "workload": "BASELINE config 5: 4B-row multi-column int32 table row-partitioned "
                    "across 1/2/4/8 B200: select+fetch+sum/min/max with NCCL allreduce",
        "total_rows": TOTAL_ROWS, "shards": N_SHARDS, "rows_per_shard": TOTAL_ROWS // N_SHARDS,
        "rows_per_step": rows_per_step, "selectivity": args.selectivity,
        "columns": "col1 uniform [0,2^30) (select), col2 uniform [2^31-10000,2^31) (fetch)",
        "l2": "inputs exceed L2 (>= 2 GB per shard column vs 126 MB)",
    }


# ------------------------------------------------------------------------------------------
# engine arm
# ------------------------------------------------------------------------------------------
def run_engine(args):
    import torch
    import analytical_database_b200 as adb
    from analytical_database_b200.engine import AGG_BYTES

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        # host-side barrier for the legs one rank runs alone (an NCCL barrier would park a
        # spinning kernel on the GPUs that rank is measuring)
        args.gloo = dist.new_group(backend="gloo")
    eng = adb.Engine(local)
    stream = torch.cuda.Stream()
    eng.set_stream(stream.cuda_stream)          # engine kernels and NCCL share one stream
    torch.cuda.set_stream(stream)

    if dist is not None and args.exchange == "peer":
        eng.peer_setup(dist)                    # map every rank's aggregate mailbox (NVLink P2P)
    if dist is None and args.exchange_self:     # debug: the exchange kernel variant at world size 1
        hbuf = C.create_string_buffer(64)
        eng._ck(eng.lib.adb_peer_create(1, 0, hbuf))
        eng._ck(eng.lib.adb_peer_connect(hbuf.raw))

    lo, hi = predicate(args.selectivity)
    shard_rows = TOTAL_ROWS // N_SHARDS
    my_shards = [s for s in range(N_SHARDS) if s % world == rank] if world > 1 else list(range(N_SHARDS))
    if args.shards_limit:
        my_shards = my_shards[:args.shards_limit]
    # ---- load: columns become HBM-resident int32 arrays -------------------------------
    cols = []
    for s in my_shards:
        c1 = eng.synth_uniform(shard_rows, SEED, s * shard_rows, 0, SPAN)
        c2 = eng.synth_uniform(shard_rows, SEED + 1, s * shard_rows, FETCH_LO, FETCH_SPAN)
        cols.append((c1, c2))
    cap = int(shard_rows * min(1.0, args.selectivity * 1.5 + 0.001)) + 4096
    # one (pos, val, count) result set per shard: every handle stays materialised
    res = [(eng.alloc_i32(cap), eng.alloc_i32(cap), eng.alloc(8)) for _ in my_shards]
    parts = eng.alloc(AGG_BYTES * max(len(my_shards), 1))
    # the allreduce operands live in torch tensors (plumbing for NCCL)
    t_sum = torch.zeros(2, dtype=torch.int64, device="cuda")      # {sum, count}
    t_mm = torch.zeros(2, dtype=torch.int32, device="cuda")       # {max, ~min}
    combined = eng.alloc(AGG_BYTES)
    blo, bhi = C.c_int32(lo), C.c_int32(hi)
    lib = eng.lib
    AggP = eng.agg_ptr

    def step(mark_base=None):
        fused_exchange = (dist is not None and args.exchange == "peer") or (dist is None and args.exchange_self)
        for i, (c1, c2) in enumerate(cols):
            pos, val, cnt = res[i]
            if mark_base is not None:
                eng._ck(lib.adb_chain_marks(mark_base + 3 * i))
            # predicate pass + expansion with the gather and the aggregates fused in; the
            # position list and the fetched vector are still materialised (pos, val)
            if fused_exchange and i == len(cols) - 1:
                # the rank's last shard: the CTA that completes its aggregate also folds the
                # earlier shards' partials and swaps the result with every peer over NVLink
                # peer memory, inside the same kernel (csrc/peer_agg.cu, adb_common.cuh)
                eng._ck(lib.adb_chain_select_fetch_agg_exchange(
                    c1.i32(), c2.i32(), shard_rows, C.byref(blo), C.byref(bhi), pos.i32(), val.i32(),
                    cnt.i64(), AggP(parts), len(cols), AggP(combined)))
            else:
                eng._ck(lib.adb_chain_select_fetch_agg(c1.i32(), c2.i32(), shard_rows, C.byref(blo),
                                                       C.byref(bhi), pos.i32(), val.i32(), cnt.i64(),
                                                       AggP(parts, i)))
        if fused_exchange:
            pass
        elif dist is None:
            eng._ck(lib.adb_agg_combine(AggP(parts), len(cols), AggP(combined), None))
        else:
            eng._ck(lib.adb_agg_combine(AggP(parts), len(cols), AggP(combined), None))
            eng._ck(lib.adb_agg_export(AggP(combined), C.c_void_p(t_sum.data_ptr()),
                                       C.c_void_p(t_mm.data_ptr())))
            dist.all_reduce(t_sum, op=dist.ReduceOp.SUM)
            dist.all_reduce(t_mm, op=dist.ReduceOp.MAX)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    # CUDA events between the chain's two launches give the live per-kernel times for the
    # roofline object, but an event record between two kernels also keeps the second one from
    # being scheduled while the first drains (programmatic dependent launch), so only every
    # fourth timed step carries them
    marks_per_step = 3 * len(cols)
    MARK_EVERY = 4
    marked_steps = [k for k in range(args.steps) if k % MARK_EVERY == 0]
    timed_marks = len(marked_steps) * marks_per_step <= 8000
    launches0 = eng.launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for k in range(args.steps):
        step((k // MARK_EVERY) * marks_per_step if timed_marks and k % MARK_EVERY == 0 else None)
    e1.record(stream)
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    launches = eng.launch_count() - launches0
    if dist is not None:
        t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        lt = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt.item())
    rows_step = shard_rows * (len(my_shards) * world if args.shards_limit else N_SHARDS)
    ms_step = ms_total / args.steps
    value = rows_step / (ms_step * 1e-3)

    # ---- result of the last step (device-resident) -----------------------------------------
    if dist is not None and args.exchange == "nccl":
        g_sum, g_cnt = int(t_sum[0].item()), int(t_sum[1].item())
        g_max, g_min = int(t_mm[0].item()), ~int(t_mm[1].item())
    else:
        a = eng.read_agg(combined)
        g_sum, g_cnt, g_min, g_max = a.sum, a.count, a.min, a.max
        if g_cnt < 0:                               # the exchange gave up on a peer (2 s): not a result
            raise SystemExit(f"rank {rank}: the aggregate exchange timed out waiting for a peer (count = -1)")

    # ---- roofline of the dominant kernel (mask_kernel: the predicate pass over the selected
    # column), from CUDA events recorded on the engine stream inside the timed region -------
    peak, peak_src = measured_peak()
    hits_local = [int(r[2].to_host(1, np.int64)[0]) for r in res]
    par = chain_parity(eng, my_shards, res, shard_rows, lo, hi)     # before anything reuses `res`
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, my_shards, res, (g_sum, g_cnt, g_min, g_max), rank)
    mask_ms, fused_ms = [], []
    if timed_marks:
        for k in range(len(marked_steps)):
            for i in range(len(cols)):
                b = k * marks_per_step + 3 * i
                mask_ms.append(eng.mark_elapsed(b, b + 1))
                fused_ms.append(eng.mark_elapsed(b + 1, b + 2))
    roofline = None
    if mask_ms:
        avg_ms = float(np.mean(mask_ms))
        alg_bytes = 4.0 * shard_rows                     # SURVEY.md 8d: the 4N of select's 4N + 4H
        achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "select_kernel_traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        h_avg = float(np.mean(hits_local))
        f_ms = float(np.mean(fused_ms))
        roofline = {"bound": "hbm", "kernel": "adb::mask_kernel (predicate pass of adb_select_scan / "
                    "adb_chain_select_fetch_agg: column -> 1 bit/row bitmap + per-chunk counts)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "frac_of_nominal_8tbs": achieved / NOMINAL_GBS,
                    "traffic": traffic, "peak_source": peak_src, "avg_launch_ms": avg_ms,
                    "algorithmic_bytes_per_launch": alg_bytes,
                    "share_of_step": float(np.mean(mask_ms) * len(cols) / ms_step),
                    "second_kernel": {
                        "kernel": "adb::expand_kernel<false,true> (bitmap -> positions, gather, "
                                  "sum/min/max fused)",
                        "avg_launch_ms": f_ms, "share_of_step": float(f_ms * len(cols) / ms_step),
                        "algorithmic_bytes_per_launch": 16.0 * h_avg,
                        "achieved": 16.0 * h_avg / (f_ms * 1e-3) / 1e9,
                        "miss_granular_bytes_per_launch": 64.0 * h_avg + 8.0 * h_avg + shard_rows / 8.0,
                        "note": "a sparse gather moves 64 bytes per hit with ld.global.nc.L2::64B "
                                "(128 with a plain load; profiles/r01c_gather_probe.md): the kernel's "
                                "DRAM traffic is about 5x its algorithmic bytes, and at 5 M random "
                                "reads per launch it runs at the DRAM random-access rate"}}
    chain_bytes = 4.0 * rows_step + 20.0 * g_cnt
    chain_gbs = chain_bytes / (ms_step * 1e-3) / 1e9

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": max(world, 1),
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int32 (int64 accumulate)", "data": "synthetic",
            "config": workload_config(args, rows_step),
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
            "chain": {"algorithmic_bytes_per_step": chain_bytes, "achieved_gbs": chain_gbs,
                      "frac_of_aggregate_peak": chain_gbs / (peak * max(world, 1)),
                      "frac_of_nominal": chain_gbs / (NOMINAL_GBS * max(world, 1)),
                      "nominal_gbs_per_gpu": NOMINAL_GBS,
                      "formula": "4N + 20H (SURVEY.md 8d)"},
            "result": {"sum": g_sum, "count": g_cnt, "min": g_min, "max": g_max},
        }
        if world > 1:
            line["config"]["aggregate_exchange"] = (
                "adb_chain_select_fetch_agg_exchange: the chain kernel of the rank's last shard folds the partials and exchanges them over NVLink peer memory (no separate launch, no NCCL call)"
                if args.exchange == "peer" else "adb_agg_export + 2 NCCL all-reduces")

    # ---- the same chain with NEITHER handle materialised (SURVEY.md 8f rank 3: 4N + 4H bytes):
    # one kernel per shard scans col1 and gathers + folds col2 at every hit; the partials meet in
    # the same exchange.  This is what the operator API runs when s and f are never read (e2e).
    lazy = None
    if not args.no_lazy:
        lz_parts = eng.alloc(AGG_BYTES * max(len(my_shards), 1))
        lz_out = eng.alloc(AGG_BYTES)

        def lazy_step():
            for i, (c1, c2) in enumerate(cols):
                eng._ck(lib.adb_chain_select_agg(c1.i32(), c2.i32(), shard_rows, C.byref(blo), C.byref(bhi),
                                                 res[i][2].i64(), AggP(lz_parts, i), None))
            if dist is not None and args.exchange == "peer":
                eng._ck(lib.adb_agg_combine_allreduce(AggP(lz_parts), len(cols), AggP(lz_out), None))
            else:
                eng._ck(lib.adb_agg_combine(AggP(lz_parts), len(cols), AggP(lz_out), None))
        for _ in range(3):
            lazy_step()
        barrier()
        z0, z1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        z0.record(stream)
        for _ in range(args.steps):
            lazy_step()
        z1.record(stream)
        barrier()
        lz_ms = z0.elapsed_time(z1) / args.steps
        la = eng.read_agg(lz_out)
        lz_sum, lz_cnt = la.sum, la.count
        if dist is not None:
            t = torch.tensor([lz_ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            lz_ms = float(t.item())
            if args.exchange != "peer":
                t2 = torch.tensor([lz_sum, lz_cnt], dtype=torch.int64, device="cuda")
                dist.all_reduce(t2, op=dist.ReduceOp.SUM)
                lz_sum, lz_cnt = int(t2[0].item()), int(t2[1].item())
        if (lz_sum, lz_cnt) != (g_sum, g_cnt) and not args.shards_limit:
            raise SystemExit(f"PARITY FAILURE: unmaterialised chain {(lz_sum, lz_cnt)} != materialised {(g_sum, g_cnt)}")
        lz_bytes = 4.0 * rows_step + 4.0 * g_cnt
        lz_gbs = lz_bytes / (lz_ms * 1e-3) / 1e9
        lazy = {"value": rows_step / (lz_ms * 1e-3), "unit": UNIT, "ms_per_step": lz_ms,
                "algorithmic_bytes_per_step": lz_bytes, "formula": "4N + 4H (SURVEY.md 8f rank 3)",
                "achieved_gbs": lz_gbs, "frac_of_aggregate_peak": lz_gbs / (peak * max(world, 1)),
                "frac_of_nominal": lz_gbs / (NOMINAL_GBS * max(world, 1)),
                "kernel": "adb::scan_gather_agg_kernel (adb_chain_select_agg): predicate pass with the gather "
                          "and the aggregates fused in, nothing written",
                "equals_materialised_chain": True}
        if rank == 0:
            line["chain_unmaterialised"] = lazy

    # ---- selectivity sweep on one shard (SURVEY.md 8d lists 0.1 %, 1 %, 10 %, 50 %) -----------
    if rank == 0 and not args.no_sweep:
        sweep = {}
        c1, c2 = cols[0]
        for sel in (0.001, 0.01, 0.1, 0.5):
            slo, shi = predicate(sel)
            need = int(shard_rows * min(1.0, sel * 1.05 + 0.001)) + 4096
            sp, sv = eng.alloc_i32(need), eng.alloc_i32(need)
            b1, b2 = C.c_int32(slo), C.c_int32(shi)

            def one():
                eng._ck(lib.adb_chain_select_fetch_agg(c1.i32(), c2.i32(), shard_rows, C.byref(b1),
                                                       C.byref(b2), sp.i32(), sv.i32(), res[0][2].i64(),
                                                       AggP(parts, 0)))
            for _ in range(2):
                one()
            eng.timer_start()
            for _ in range(5):
                one()
            ms = eng.timer_stop() / 5
            h = int(res[0][2].to_host(1, np.int64)[0])
            gbs = (4.0 * shard_rows + 20.0 * h) / (ms * 1e-3) / 1e9
            sweep[str(sel)] = {"ms_per_shard": ms, "hits": h, "rows_per_s_per_gpu": shard_rows / (ms * 1e-3),
                               "chain_algorithmic_gbs": gbs, "frac_of_peak": gbs / peak}
            sp.free()
            sv.free()
        line["selectivity_sweep"] = sweep

    # second half of BASELINE.json's metric: hash-join tuples/s (config 4).  N > 1: both tables
    # row-range sharded, pairs hash-routed to their owners, joined locally.
    join_sharded = None
    if world > 1 and args.join_torch:
        join_sharded = measure_join_sharded(eng, dist, rank, world, local, args.gloo)

    # ---- parity at every N: each rank diffs a window of every shard it owns -- positions and
    # fetched values of the last timed step -- against the reference's operators run on the same
    # rows regenerated on the host (numpy twin of the generator), and the table-wide aggregate
    # against the N-independent constants of the synthetic table
    if dist is not None:
        t = torch.tensor([1 if par["ok"] else 0], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        par["ok"] = bool(t.item())
    if rank == 0:
        line["parity"] = {"chain": par["ok"], "chain_detail": par["detail"],
                          "join": (join_sharded or {}).get("parity")}
    if not par["ok"]:
        raise SystemExit(f"PARITY FAILURE (rank {rank}): {par}")
    if join_sharded is not None and join_sharded.get("parity") is False:
        raise SystemExit(f"PARITY FAILURE in the sharded join (rank {rank})")

    # ---- e2e (one host process drives all N GPUs) and cpu_baseline (the CPU leg only at N = 1)
    e2e = measure_e2e(args, eng, cols, shard_rows, lo, hi, world, dist, rank, (g_sum, g_cnt))
    if rank == 0:
        cold = e2e.pop("cold", None)
        for k_, v_ in (e2e.pop("configs", None) or {}).items():
            line[k_] = v_
        aj = e2e.pop("api_join", None)
        if aj is not None and "error" not in aj:
            line["hash_join"] = join_summary(aj, max(world, 1))
            line["hash_join"]["through"] = "the operator API (host/query_shim.c), one host process"
            if "parity" in line:
                line["parity"]["join"] = aj.get("parity")
        elif aj is not None:
            line["hash_join"] = aj
        line["e2e"] = e2e
        if cold is not None:
            line["e2e_cold"] = cold
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = measure_cpu(args, eng, cols, res, shard_rows, lo, hi)
        if world == 1 and (args.ops or not args.no_join):
            for c1, c2 in cols[1:]:
                c1.free()
                c2.free()
        if world == 1 and args.join_torch and not args.ops:
            line["hash_join_c_abi"] = measure_join_single(args)
        if world == 1 and args.ops:
            line["ops"] = measure_ops(args)
            if "hash_join_100Mx100M" in line["ops"]:
                line["hash_join"] = join_summary(line["ops"]["hash_join_100Mx100M"], 1)
        if world > 1 and join_sharded is not None:
            line["hash_join_process_per_gpu"] = join_summary(join_sharded, world)
        emit(line)
    barrier()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def chain_parity(eng, my_shards, res, shard_rows, lo, hi, window=1 << 22):
    """Oracle check of what the timed chain left in HBM, on this rank's shards: the first
    `window` rows of every shard are regenerated on the host (numpy twin of the generator) and
    run through the reference's select -> fetch (oracle/_ref when built, else the restatement);
    the GPU's position list and value vector must start with exactly those tuples."""
    from analytical_database_b200 import synth
    ops, kind, _ = cpu_ops()
    ok, checked = True, 0
    for i, s_ in enumerate(my_shards):
        pos, val, cnt = res[i]
        h = int(cnt.to_host(1, np.int64)[0])
        sel = synth.uniform(window, SEED, s_ * shard_rows, 0, SPAN)
        fet = synth.uniform(window, SEED + 1, s_ * shard_rows, FETCH_LO, FETCH_SPAN)
        epos = ops.select_scan(sel, lo, hi)
        evals = ops.fetch(fet, epos)
        k = epos.size
        gpos, gval = pos.to_host(min(h, k + 1)), val.to_host(min(h, k + 1))
        good = h >= k and np.array_equal(gpos[:k], epos) and np.array_equal(gval[:k], evals) and \
            (h == k or gpos[k] >= window)
        ok = ok and bool(good)
        checked += k
    return {"ok": ok, "detail": f"{len(my_shards)} shards x first {window} rows vs {kind}: {checked} tuples"}


def dump_outputs(out_dir, my_shards, res, agg, rank):
    """What the timed chain handed its caller in its last step, as float64 .npy files (exact: every
    value is an integer below 2^53).  Per shard: `shard<s>_hits` (the length of the position list)
    and `shard<s>_positions` / `shard<s>_values`, the entries of the position list and of the
    fetched vector at DUMP_SAMPLE indices drawn with a seed fixed per shard (the whole lists when
    they are shorter).  Rank 0 adds `aggregate`: [sum >> 32, sum & 0xffffffff, count, min, max]."""
    os.makedirs(out_dir, exist_ok=True)
    for i, s_ in enumerate(my_shards):
        pos, val, cnt = res[i]
        h = int(cnt.to_host(1, np.int64)[0])
        idx = np.arange(h)
        if h > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(SEED + s_).choice(h, DUMP_SAMPLE, replace=False))
        np.save(os.path.join(out_dir, f"shard{s_}_hits.npy"), np.array([h], np.float64))
        np.save(os.path.join(out_dir, f"shard{s_}_positions.npy"), pos.to_host(h)[idx].astype(np.float64))
        np.save(os.path.join(out_dir, f"shard{s_}_values.npy"), val.to_host(h)[idx].astype(np.float64))
    if rank == 0:
        g_sum, g_cnt, g_min, g_max = agg
        np.save(os.path.join(out_dir, "aggregate.npy"),
                np.array([g_sum >> 32, g_sum & 0xFFFFFFFF, g_cnt, g_min, g_max], np.float64))


def measure_e2e(args, eng, cols, shard_rows, lo, hi, world, dist, rank, expect):
    """The same chain through the reference-facing operator API -- the C host drop-in
    (host/query_shim.c -> libadb_query.so) called exactly as src/server.c:137-290 calls
    query.c: select_column(Column*, &lo, &hi) -> fetch_column(Column*, Result*) ->
    sum(GeneralizedColumn*) with host Column / Result / Status structs, every operator
    returning its num_tuples to the host before the next is issued (parse.c:799 needs it),
    the long read back from the scalar Result, and the handles released the way
    client_context.c does.  Wall clock.

    ONE process (rank 0) drives all N GPUs, as the reference's one-process server would
    (adb_host_init_multi): the table is E2E_PARTS columns of E2E_PART_ROWS rows, every column
    row-range sharded over the N GPUs by the shim; a select fans out over the shards, the
    aggregate's partials meet in one exchange over NVLink peer memory inside the kernel that
    produces them, and the host reads one Result per operator.  The other ranks idle at a host
    barrier meanwhile.

    warm: a table is in HBM once loaded (the reference keeps loaded columns in RAM the same
          way); the timed steps then move only the bounds down and the counts / sum up.
    cold: one shard whose two columns live in HOST memory and are invalidated before every
          step, so each step pays the H2D copy of 2 x 2 GB inside the timed region (N = 1)."""
    if rank != 0:
        dist.barrier(group=args.gloo)           # rank 0 is measuring; wait on the host
        return None
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import query_api as q                      # ctypes view of include/adb_query_api.h
    api = q.Api()
    L = api.lib
    G = max(world, 1)
    if L.adb_host_init_multi(G) != 0:
        raise SystemExit("adb_host_init_multi: " + L.adb_host_last_error().decode())
    lib = eng.lib
    S = E2E_PART_ROWS // G
    assert S % 32 == 0 and S * G == E2E_PART_ROWS and E2E_PARTS * E2E_PART_ROWS == TOTAL_ROWS
    bufs, hcols = [], []
    for p_ in range(E2E_PARTS):
        pa, pb = (C.c_void_p * G)(), (C.c_void_p * G)()
        for g in range(G):
            eng._ck(lib.adb_ctx_select(g))
            first = p_ * E2E_PART_ROWS + g * S
            b1 = eng.synth_uniform(S, SEED, first, 0, SPAN)
            b2 = eng.synth_uniform(S, SEED + 1, first, FETCH_LO, FETCH_SPAN)
            eng.sync()
            bufs += [(g, b1), (g, b2)]
            pa[g], pb[g] = b1.ptr, b2.ptr
        eng._ck(lib.adb_ctx_select(0))
        a, b = q.Column(), q.Column()
        a.name, b.name = b"col1", b"col2"
        a.row_count = b.row_count = E2E_PART_ROWS
        assert L.adb_host_column_adopt_shards(C.byref(a), pa, S) == 0, L.adb_host_last_error()
        assert L.adb_host_column_adopt_shards(C.byref(b), pb, S) == 0, L.adb_host_last_error()
        hcols.append((a, b))
    blo, bhi = C.c_int(lo), C.c_int(hi)
    st = q.Status(99, None)
    gen = q.GeneralizedColumn(q.RESULT)

    def chain(a, b):
        s_ = L.select_column(C.byref(a), C.byref(blo), C.byref(bhi), C.byref(st))
        if st.code != q.OK:
            raise SystemExit("select_column: " + L.adb_host_last_error().decode())
        f_ = L.fetch_column(C.byref(b), s_, C.byref(st))
        gen.column_pointer.result = f_
        r_ = L.sum(C.byref(gen), C.byref(st))
        if st.code != q.OK:
            raise SystemExit("fetch/sum: " + L.adb_host_last_error().decode())
        total = C.cast(r_.contents.payload, C.POINTER(C.c_long))[0]
        hits = s_.contents.num_tuples
        trio[0], trio[1], trio[2] = s_, f_, r_
        L.adb_host_results_drop(trio, 3)        # what free_client_context does per handle
        return total, hits

    trio = (q.RP * 3)()

    def step():
        tot = hits = 0
        for (a, b) in hcols:
            t_, h_ = chain(a, b)
            tot += t_
            hits += h_
        return tot, hits

    def sync_all():
        for g in range(G):
            lib.adb_ctx_select(g)
            eng.sync()
        lib.adb_ctx_select(0)

    # The timed loop is the dispatcher's sequence written in C (host/api_harness.c ->
    # libadb_harness.so: select_column -> fetch_column -> sum -> release, exactly chain() above):
    # the operators are called from C in the reference, and ctypes costs ~2 us per call.
    H = C.CDLL(os.path.join(ROOT, "analytical-database_b200", "libadb_harness.so"))
    H.adb_harness_select_fetch_sum.restype = C.c_int
    H.adb_harness_select_fetch_sum.argtypes = [C.POINTER(C.POINTER(q.Column)), C.POINTER(C.POINTER(q.Column)), C.c_int,
                                               C.c_int, C.c_int, C.c_int, C.POINTER(C.c_long),
                                               C.POINTER(C.c_size_t), C.POINTER(C.c_double)]
    sel_arr = (C.POINTER(q.Column) * len(hcols))(*[C.pointer(a) for a, _ in hcols])
    fet_arr = (C.POINTER(q.Column) * len(hcols))(*[C.pointer(b) for _, b in hcols])
    steps = args.steps
    l0 = lib.adb_launch_count_all()
    tot_py, hits_py = step()                    # the Python spelling of the same chain, once
    c_sum, c_hits, c_sec = C.c_long(0), C.c_size_t(0), C.c_double(0.0)

    def harness(k):
        if H.adb_harness_select_fetch_sum(sel_arr, fet_arr, len(hcols), lo, hi, k, C.byref(c_sum), C.byref(c_hits),
                                          C.byref(c_sec)) != 0:
            raise SystemExit("e2e harness: " + L.adb_host_last_error().decode())
    harness(2)
    sync_all()
    L.adb_host_profile_dump()                   # (ADB_SHIM_PROFILE=1: start the phase timers afresh)
    harness(steps)
    sync_all()
    dt = c_sec.value
    tot, hits = c_sum.value, c_hits.value
    if (tot, hits) != (tot_py, hits_py):
        raise SystemExit(f"e2e harness {(tot, hits)} != the same chain driven from Python {(tot_py, hits_py)}")
    L.adb_host_profile_dump()
    launches = (lib.adb_launch_count_all() - l0) // (steps + 3)
    rows_step = E2E_PARTS * E2E_PART_ROWS
    if (tot, hits) != tuple(expect) and not args.shards_limit:
        raise SystemExit(f"PARITY FAILURE: e2e chain {(tot, hits)} != device-resident chain {tuple(expect)}")
    out = {"value": rows_step * steps / dt, "unit": UNIT,
           "h2d_bytes_per_step": 0,
           "d2h_bytes_per_step": (8 * G + 24) * E2E_PARTS,
           "ms_per_step": 1e3 * dt / steps, "steps": steps, "gpu_launches_per_step": int(launches),
           "host_processes": 1, "gpus_driven": G,
           "caller": "host/api_harness.c (C, as the reference's dispatcher is): select_column -> fetch_column -> "
                     "sum -> release per column, wall clock around all steps",
           "api": "select_column -> fetch_column -> sum of include/adb_query_api.h (libadb_query.so = "
                  f"host/query_shim.c, adb_host_init_multi({G})): one call chain per column of "
                  f"{E2E_PART_ROWS} rows, each column row-range sharded over the {G} GPU(s) by the shim",
           "bytes_model": "4N + 4H: s and f are lazy handles (host/query_shim.c) -- the aggregate gathers and folds "
                          "the hit rows straight from the select's bitmap and neither list is written, because "
                          "the harness, like a client that only prints the sum, never reads them",
           "mode": "warm: columns HBM-resident after load; bounds travel as kernel arguments "
                   "(no H2D copy); per column the host reads every shard's num_tuples (8 B) after select "
                   "and the exchanged aggregate (24 B) after sum; wall clock; see `e2e_cold` for the "
                   "H2D-inclusive figure",
           "check": {"sum": tot, "hits": hits, "equals_device_resident_chain": True}}
    for (a, b) in hcols:
        L.adb_host_column_invalidate(C.byref(a))
        L.adb_host_column_invalidate(C.byref(b))
    for g, b in bufs:
        lib.adb_ctx_select(g)
        b.free()
    lib.adb_ctx_select(0)
    # BASELINE configs 2 and 3 through the same operator API and the same G GPUs
    if not args.no_configs:
        try:
            out["configs"] = {"config2_shared_scan": api_shared_scan(eng, api, q, G, sync_all),
                              "config3_index": api_index(eng, api, q, G, sync_all)}
        except Exception as e:                              # the headline line must survive
            out["configs"] = {"error": repr(e)}
    if not args.no_join:
        try:
            out["api_join"] = api_join(eng, api, q, G, sync_all)
        except Exception as e:
            out["api_join"] = {"error": repr(e)}
    # cold: HOST columns, re-uploaded by the shim inside every timed step
    if world == 1 and not args.no_cold:
        c1, c2 = cols[0]
        h1, h2 = c1.to_host(shard_rows), c2.to_host(shard_rows)

        def host_col(host):
            c = q.Column()
            c.name = b"col"
            c.row_count = shard_rows
            c.data = host.ctypes.data_as(C.POINTER(C.c_int))
            return c
        a, b = host_col(h1), host_col(h2)
        chain(a, b)                                         # first touch
        L.adb_host_column_invalidate(C.byref(a))            # second upload of the same arrays: the shim
        L.adb_host_column_invalidate(C.byref(b))            # page-locks them once (as it would for a column
        chain(a, b)                                         # that insert_row keeps invalidating)
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            L.adb_host_column_invalidate(C.byref(a))
            L.adb_host_column_invalidate(C.byref(b))
            ctot, chits = chain(a, b)
        dtc = time.perf_counter() - t0
        L.adb_host_column_invalidate(C.byref(a))
        L.adb_host_column_invalidate(C.byref(b))
        out["cold"] = {"value": shard_rows * reps / dtc, "unit": UNIT,
                       "h2d_bytes_per_step": 8 * shard_rows, "d2h_bytes_per_step": 32,
                       "ms_per_step": 1e3 * dtc / reps,
                       "sample": f"one {shard_rows}-row shard whose two columns are host arrays; the "
                                 "shim uploads both inside every timed step (the arrays were page-locked by "
                                 "the shim at their second upload, outside the timed region: one DMA per "
                                 "column at the link's rate; a first upload goes through the engine's pinned "
                                 "multi-lane staging pipeline)",
                       "check": {"sum": ctot, "hits": chits}}
    if dist is not None:
        dist.barrier(group=args.gloo)
    return out


def adopt_sharded(eng, api, q, G, rows, fill, name, **flags):
    """A Column of `rows` rows whose shards are generated on the GPUs (fill(g, first_row, count) ->
    DevBuf on the current context) and adopted by the shim (no host copy)."""
    lib, L = eng.lib, api.lib
    S = ((rows + G - 1) // G + 31) // 32 * 32
    ptrs, bufs = (C.c_void_p * G)(), []
    for g in range(G):
        eng._ck(lib.adb_ctx_select(g))
        cnt = max(0, min(S, rows - g * S))
        b = fill(g, g * S, max(cnt, 1))
        eng.sync()
        bufs.append((g, b))
        ptrs[g] = b.ptr
    eng._ck(lib.adb_ctx_select(0))
    col = q.Column()
    col.name = name
    col.row_count = rows
    for k, v in flags.items():
        setattr(col, k, v)
    assert L.adb_host_column_adopt_shards(C.byref(col), ptrs, S) == 0, L.adb_host_last_error()
    return col, bufs


def free_sharded(eng, api, col, bufs):
    api.lib.adb_host_column_invalidate(C.byref(col))
    for g, b in bufs:
        eng.lib.adb_ctx_select(g)
        b.free()
    eng.lib.adb_ctx_select(0)


def api_shared_scan(eng, api, q, G, sync_all, n=100_000_000, nq=100):
    """BASELINE config 2: 100 concurrent range selects over a 100 M-row column in one
    shared_select call of the operator API (query.h:36; the dispatcher's batch_execute,
    server.c:366-393), the column row-range sharded over the G GPUs."""
    from analytical_database_b200 import synth
    L = api.lib
    peak, _ = measured_peak()
    col, bufs = adopt_sharded(eng, api, q, G, n, lambda g, first, cnt: eng.synth_uniform(cnt, SEED, first, 0, n), b"c2")
    rng = np.random.default_rng(SEED)
    lows = rng.integers(0, n - n // 1000, nq).astype(np.int32)
    highs = (lows + n // 1000).astype(np.int32)
    ops = (q.SelectOperator * nq)()
    for k in range(nq):
        ops[k].low, ops[k].high, ops[k].has_low, ops[k].has_high = int(lows[k]), int(highs[k]), 1, 1
    st = q.Status(99, None)

    def run(keep=False):
        res = L.shared_select(ops, nq, C.byref(col), C.byref(st))
        if st.code != q.OK or not res:
            raise RuntimeError("shared_select: " + L.adb_host_last_error().decode())
        if not keep:                            # timed form: the batch's handles go the way
            L.adb_host_results_drop(res, nq)    # free_client_context releases them
            q._libc.free(C.cast(res, C.c_void_p))
            return None, None
        hs = [res[k].contents.num_tuples for k in range(nq)]
        handles = [C.pointer(res[k].contents) for k in range(nq)]
        q._libc.free(C.cast(res, C.c_void_p))
        if keep:
            return hs, handles
        for h_ in handles:
            api.drop(h_)
        return hs, None
    for _ in range(2):
        run()
    sync_all()
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        run()
    sync_all()
    ms = 1e3 * (time.perf_counter() - t0) / reps
    # oracle window: the first 4 M rows regenerated on the host, ten of the queries
    hs, handles = run(keep=True)
    cpu, kind, _ = cpu_ops()
    W = 1 << 22
    win = synth.uniform(W, SEED, 0, 0, n)
    ok = True
    for k in range(0, nq, 10):
        exp = cpu.select_scan(win, int(lows[k]), int(highs[k]))
        got = api.tuples(handles[k])
        ok = ok and got.size >= exp.size and np.array_equal(got[:exp.size], exp) and \
            (got.size == exp.size or got[exp.size] >= W) and bool(np.all(np.diff(got) > 0))
    for h_ in handles:
        api.drop(h_)
    free_sharded(eng, api, col, bufs)
    alg = 4.0 * n + 4.0 * sum(hs)
    if not ok:
        raise SystemExit("PARITY FAILURE: shared_select window differs from the reference")
    return {"rows": n, "queries": nq, "hits": int(sum(hs)), "ms": ms, "gpus": G,
            "rows_per_s": n / (ms * 1e-3), "pred_evals_per_s": n * nq / (ms * 1e-3),
            "algorithmic_bytes": alg, "formula": "4N + 4*sum(H_q)", "alg_gbs": alg / (ms * 1e-3) / 1e9,
            "frac_of_peak": alg / (ms * 1e-3) / 1e9 / (peak * G),
            "frac_of_nominal": alg / (ms * 1e-3) / 1e9 / (NOMINAL_GBS * G),
            "through": "shared_select of include/adb_query_api.h: one slab per GPU, one Result per query; "
                       "wall clock incl. the host reading all counts",
            "parity": f"first {W} rows x 10 queries vs {kind} + ascending order of every checked list"}


def api_index(eng, api, q, G, sync_all, n=500_000_000):
    """BASELINE config 3: index build + range select + fetch over 500 M rows through the operator
    API.  The indexed key is a permutation of 0..n-1 (unique keys: any correct sort equals the
    reference's, SURVEY.md A3 / 8d), (row * mul + add) mod n, so the oracle is a closed form: the
    row holding key v is inv(mul) * (v - add) mod n -- checked against the reference's own index
    build in tests/test_gpu_index_build.py."""
    from analytical_database_b200 import synth
    L, lib = api.lib, eng.lib
    peak, _ = measured_peak()
    mul, add = 387_420_489, 123_456_789              # 3^18: coprime with n = 2^8 * 5^9 * ...
    import math
    assert math.gcd(mul, n) == 1
    inv = pow(mul, -1, n)

    def fill_key(g, first, cnt):
        b = eng.alloc_i32(cnt)
        eng._ck(lib.adb_synth_affine(b.i32(), cnt, first, mul, add, n))
        return b
    key, kb = adopt_sharded(eng, api, q, G, n, fill_key, b"key", has_index=True, sorted=False, clustered=False)
    pay, pb = adopt_sharded(eng, api, q, G, n, lambda g, first, cnt: eng.synth_uniform(cnt, 8, first, 0, 10000), b"pay")
    arr = (C.POINTER(q.Column) * 2)(C.pointer(key), C.pointer(pay))
    sync_all()
    t0 = time.perf_counter()
    if L.adb_host_index_build(arr, 2, 0) != 0:
        raise RuntimeError("adb_host_index_build: " + L.adb_host_last_error().decode())
    build_s = time.perf_counter() - t0
    out = {"rows": n, "gpus": G, "index": "btree, unclustered (B+-tree descent + sorted-array slices, "
           "range-partitioned by index order over the GPUs)",
           "build_s_incl_host_copy": build_s,
           "build_note": "adb_host_index_build: engine radix sort + 6 GB of (values, size_t positions) copied "
                         "back into the catalog's host arrays, which the unchanged plumbing persists"}
    hv = np.ctypeslib.as_array(key.index.contents.values, shape=(n,))
    hp = np.ctypeslib.as_array(key.index.contents.positions, shape=(n,))
    ok = bool(np.array_equal(hv[:1 << 20], np.arange(1 << 20, dtype=np.int32)))
    vs = np.arange(n - (1 << 20), n, dtype=np.int64)
    ok = ok and bool(np.array_equal(hp[n - (1 << 20):], ((vs - add) % n * inv % n).astype(np.uint64)))
    st = q.Status(99, None)
    cases = {}
    for sel in (0.0002, 0.01, 0.1):
        lo = n // 7
        hi = lo + int(n * sel)
        blo, bhi = C.c_int(lo), C.c_int(hi)

        def run(keep=False):
            s_ = L.select_column(C.byref(key), C.byref(blo), C.byref(bhi), C.byref(st))
            if st.code != q.OK:
                raise RuntimeError("select_column: " + L.adb_host_last_error().decode())
            f_ = L.fetch_column(C.byref(pay), s_, C.byref(st))
            if st.code != q.OK:
                raise RuntimeError("fetch_column: " + L.adb_host_last_error().decode())
            h = s_.contents.num_tuples
            if keep:
                return h, s_, f_
            api.drop(s_)
            api.drop(f_)
            return h, None, None
        for _ in range(2):
            run()
        sync_all()
        reps = 5
        t0 = time.perf_counter()
        for _ in range(reps):
            h, _, _ = run()
        sync_all()
        ms = 1e3 * (time.perf_counter() - t0) / reps
        # oracle: the first and last 2^20 tuples of the value-ordered result
        h, s_, f_ = run(keep=True)
        gpos, gval = api.tuples(s_), api.tuples(f_)
        W = min(h, 1 << 20)
        for a0 in (0, h - W):
            vs = np.arange(lo + a0, lo + a0 + W, dtype=np.int64)
            epos = ((vs - add) % n * inv % n).astype(np.int32)
            z = synth.mix64(8, epos.astype(np.uint64))
            evals = (((z >> np.uint64(32)) * np.uint64(10000)) >> np.uint64(32)).astype(np.int32)
            ok = ok and h == hi - lo and bool(np.array_equal(gpos[a0:a0 + W], epos)) and \
                bool(np.array_equal(gval[a0:a0 + W], evals))
        api.drop(s_)
        api.drop(f_)
        alg = 8.0 * h + 12.0 * h
        cases[f"sel_{sel}"] = {"hits": int(h), "ms": ms, "algorithmic_bytes": alg,
                               "formula": "select 4H (int32 index positions) + 4H out, fetch 12H",
                               "alg_gbs": alg / (ms * 1e-3) / 1e9,
                               "frac_of_peak": alg / (ms * 1e-3) / 1e9 / (peak * G),
                               "gathers_per_s": h / (ms * 1e-3)}
    out["cases"] = cases
    out["parity"] = "index arrays + first/last 2^20 tuples of every result (positions and fetched values) vs the closed form of the permutation"
    ix = key.index.contents
    q._libc.free(C.cast(ix.values, C.c_void_p))
    q._libc.free(C.cast(ix.positions, C.c_void_p))
    q._libc.free(C.cast(key.index, C.c_void_p))
    key.index = None
    free_sharded(eng, api, key, kb)
    free_sharded(eng, api, pay, pb)
    if not ok:
        raise SystemExit("PARITY FAILURE: index select / fetch differs from the closed-form oracle")
    return out


def api_join(eng, api, q, G, sync_all, n=100_000_000):
    """BASELINE config 4 through the operator API: two 100 M-row tables (key uniform in [1, n],
    filter column uniform in [0, 1000)), prefilter select(f, null, x) + fetch(k, .) on each side,
    then hash_join(v1, p1, v2, p2) of the reference's query.h -- ONE call that, with G > 1,
    hash-partitions the build side over the GPUs through peer memory and probes every GPU's slice
    of the probe side in place (host/query_shim.c join_sharded).  Output order is the
    reference's (probe-major), checked element for element on a 2 M-row instance."""
    from analytical_database_b200 import synth
    L = api.lib
    cpu, kind, _ = cpu_ops()

    def tables(rows, seeds):
        cols, bufs = {}, []
        for name, seed, lo, span in (("k1", seeds[0], 1, rows), ("f1", seeds[1], 0, 1000),
                                     ("k2", seeds[2], 1, rows), ("f2", seeds[3], 0, 1000)):
            c, b = adopt_sharded(eng, api, q, G, rows,
                                 lambda g, first, cnt, s_=seed, l_=lo, sp_=span: eng.synth_uniform(cnt, s_, first, l_, sp_),
                                 name.encode())
            cols[name] = c
            bufs.append((c, b))
        return cols, bufs

    def prefiltered(cols, x1, x2):
        p1 = api.select_column(cols["f1"], None, x1)
        p2 = api.select_column(cols["f2"], None, x2)
        v1, v2 = api.fetch_column(cols["k1"], p1), api.fetch_column(cols["k2"], p2)
        return v1, p1, v2, p2

    # ---- parity: 2 M x 2 M rows, prefilters 0.8 / 0.15, pair lists element for element
    ns = 2_000_000
    cols, bufs = tables(ns, (21, 23, 22, 24))
    v1, p1, v2, p2 = prefiltered(cols, 800, 150)
    o1, o2 = api.join("hash_join", v1, p1, v2, p2)
    k1, f1 = synth.uniform(ns, 21, 0, 1, ns), synth.uniform(ns, 23, 0, 0, 1000)
    k2, f2 = synth.uniform(ns, 22, 0, 1, ns), synth.uniform(ns, 24, 0, 0, 1000)
    e1, e2 = cpu.select_scan(f1, None, 800), cpu.select_scan(f2, None, 150)
    r1, r2 = cpu.hash_join(k1[e1], e1, k2[e2], e2)
    parity = bool(np.array_equal(api.tuples(o1), r1) and np.array_equal(api.tuples(o2), r2))
    for h_ in (v1, p1, v2, p2, o1, o2):
        api.drop(h_)
    for c, b in bufs:
        free_sharded(eng, api, c, b)
    if not parity:
        raise SystemExit("PARITY FAILURE: hash_join through the operator API differs from the reference's pair lists")
    # ---- timing at full size
    cols, bufs = tables(n, (11, 13, 12, 14))
    cases = {"parity": True,
             "parity_detail": f"2M x 2M rows, prefilters 0.8 / 0.15, {r1.size} pairs element for element "
                              f"(probe-major order) vs {kind}"}
    for s1, s2 in ((0.8, 0.15), (1.0, 1.0)):
        v1, p1, v2, p2 = prefiltered(cols, int(1000 * s1), int(1000 * s2))
        api.tuples(v1)[:1], api.tuples(v2)[:1]             # the lazy handles are written before the clock starts
        ms = []
        for it in range(4):
            sync_all()
            t0 = time.perf_counter()
            o1, o2 = api.join("hash_join", v1, p1, v2, p2)
            sync_all()
            ms.append(1e3 * (time.perf_counter() - t0))
            m = o1.contents.num_tuples
            api.drop(o1)
            api.drop(o2)
        best = min(ms[1:])
        nb, np_ = v1.contents.num_tuples, v2.contents.num_tuples
        cases[f"prefilter_{s1}_{s2}"] = {
            "build": int(nb), "probe": int(np_), "matches": int(m), "ms": best, "world": G,
            "tuples_per_s": (nb + np_) / (best * 1e-3),
            "algorithmic_bytes": 8.0 * (nb + np_) + 8.0 * m, "formula": "8(B+P) + 8M (SURVEY.md 8d)",
            "alg_gbs": (8.0 * (nb + np_) + 8.0 * m) / (best * 1e-3) / 1e9,
            "includes": "hash_join of include/adb_query_api.h, wall clock: "
                        + ("build-side exchange over NVLink peer memory, per-GPU tables, probe in place with "
                           "peer table reads, output sized and written" if G > 1 else
                           "build sort + tables, probe rows partitioned by window and table slice, slice-major probe, "
                           "back to row order, expansion (offsets computed in the expansion) on one GPU")}
        for h_ in (v1, p1, v2, p2):
            api.drop(h_)
    for c, b in bufs:
        free_sharded(eng, api, c, b)
    return cases


def measure_join_sharded(eng, dist, rank, world, local, args_gloo):
    """BASELINE config 4: hash join of two 100 M-row tables with selective prefilters, both
    row-range sharded over the ranks, pairs hash-routed by key and pushed into the destination
    ranks' memory over NVLink (adb_peer_exchange_pairs), joined locally; the NCCL all-to-all-v
    exchange is timed next to it.  Returns tuples/s over all ranks (max time)."""
    import torch
    from analytical_database_b200.sharded import EngineOps, ShardedTable, shard_range
    dev = torch.device("cuda", local)
    ops = EngineOps(eng, dev)                 # engine stream = torch's current stream
    n = 100_000_000
    out = {}
    b, e = shard_range(n, rank, world)
    rows = e - b

    def col(seed, lo, span, first=None, count=None):
        first, count = (b, rows) if first is None else (first, count)
        t = torch.empty(count, dtype=torch.int32, device=dev)
        eng._ck(eng.lib.adb_synth_uniform(C.cast(C.c_void_p(t.data_ptr()), C.POINTER(C.c_int32)),
                                          count, seed, first, lo, span))
        return t
    t1 = ShardedTable(ops, {"k": col(11, 1, n), "f": col(13, 0, 1000)}, n, dist)
    t2 = ShardedTable(ops, {"k": col(12, 1, n), "f": col(14, 0, 1000)}, n, dist)
    # receive regions of the peer-memory pair exchange: 30 % head room over an even split
    ops.connect_peers(dist, join_cap_pairs=int(1.3 * n / world) + (1 << 16))

    def timed_join(v1, g1, v2, g2):
        ms = []
        for it in range(4):
            torch.cuda.synchronize()
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            o1, o2 = t1.hash_join(v1, g1, v2, g2)
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        t = torch.tensor([min(ms[1:])], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        m = torch.tensor([o1.numel()], dtype=torch.int64, device=dev)
        dist.all_reduce(m, op=dist.ReduceOp.SUM)
        return float(t.item()), int(m.item())

    # parity: the same sharded join on two 2 M-row tables, its pair set (gathered on rank 0)
    # against the reference's hash_join on the same rows regenerated on the host
    ns = 2_000_000
    sb, se = shard_range(ns, rank, world)
    s1t = ShardedTable(ops, {"k": col(21, 1, ns, sb, se - sb), "f": col(23, 0, 1000, sb, se - sb)}, ns, dist)
    s2t = ShardedTable(ops, {"k": col(22, 1, ns, sb, se - sb), "f": col(24, 0, 1000, sb, se - sb)}, ns, dist)
    q1, q2 = s1t.select("f", None, 800), s2t.select("f", None, 150)
    w1, w2 = s1t.fetch("k", q1), s2t.fetch("k", q2)
    j1, j2 = s1t.hash_join(w1, q1.local + q1.base, w2, q2.local + q2.base)
    mine = np.stack([j1.cpu().numpy(), j2.cpu().numpy()], axis=1) if j1.numel() else np.zeros((0, 2), np.int32)
    gathered = [None] * world
    dist.all_gather_object(gathered, mine, group=args_gloo)
    out["parity"] = None
    if rank == 0:
        from analytical_database_b200 import synth
        cpu, kind, _ = cpu_ops()
        k1, f1 = synth.uniform(ns, 21, 0, 1, ns), synth.uniform(ns, 23, 0, 0, 1000)
        k2, f2 = synth.uniform(ns, 22, 0, 1, ns), synth.uniform(ns, 24, 0, 0, 1000)
        e1, e2 = cpu.select_scan(f1, None, 800), cpu.select_scan(f2, None, 150)
        r1, r2 = cpu.hash_join(k1[e1], e1, k2[e2], e2)
        got = np.concatenate(gathered)
        exp = np.stack([r1, r2], axis=1)
        got = got[np.lexsort((got[:, 0], got[:, 1]))]
        exp = exp[np.lexsort((exp[:, 0], exp[:, 1]))]
        out["parity"] = bool(got.shape == exp.shape and np.array_equal(got, exp))
        out["parity_detail"] = f"2M x 2M rows, prefilters 0.8 / 0.15, {exp.shape[0]} pairs as a sorted set vs {kind}"
    flag = torch.tensor([1 if out["parity"] in (None, True) else 0], dtype=torch.int64, device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if int(flag.item()) == 0:
        out["parity"] = False

    for s1, s2 in ((0.8, 0.15), (1.0, 1.0)):
        p1, p2 = t1.select("f", None, int(1000 * s1)), t2.select("f", None, int(1000 * s2))
        v1, v2 = t1.fetch("k", p1), t2.fetch("k", p2)
        g1, g2 = p1.local + p1.base, p2.local + p2.base        # global positions (< 2^31)
        tup = p1.total + p2.total
        ops.peer_join = True
        ms_peer, m_peer = timed_join(v1, g1, v2, g2)
        ops.peer_join = False
        ms_nccl, m_nccl = timed_join(v1, g1, v2, g2)
        ops.peer_join = True
        out[f"prefilter_{s1}_{s2}"] = {
            "build": p1.total, "probe": p2.total, "matches": m_peer, "matches_equal": m_peer == m_nccl,
            "ms": ms_peer, "tuples_per_s": tup / (ms_peer * 1e-3), "world": world,
            "includes": "adb_peer_exchange_pairs for both sides (counts all-gather, routing scatter into the "
                        "destination ranks' memory over NVLink, done flags) + local join",
            "nccl_exchange": {"ms": ms_nccl, "tuples_per_s": tup / (ms_nccl * 1e-3),
                              "includes": "adb_route_pairs, 2 x (count + 2 payload) NCCL all-to-all, local join"}}
    return out


def join_summary(cases: dict, world: int) -> dict:
    """The `hash_join` object of the JSON line: tuples/s = (build + probe tuples) / time."""
    out = {"metric": "hash-join tuples/sec", "unit": "tuples/s", "n_gpus": world,
           "workload": "BASELINE config 4: 100M x 100M int32 key columns (uniform in [1, 100M]), prefilter "
                       "select(f, null, x) on each side, hash join of the (value, position) pair lists"
                       + (", pairs hash-partitioned across the ranks over NVLink" if world > 1 else ""),
           "cases": cases}
    full = cases.get("prefilter_1.0_1.0")
    if full:
        out["value"] = full["tuples_per_s"]
        out["ms"] = full["ms"]
    return out


def measure_join_single(args):
    """BASELINE config 4 on one GPU (adb_hash_join_count + adb_join_emit), two prefilter cases."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_ops
    import analytical_database_b200 as adb
    eng = adb.Engine(int(os.environ.get("LOCAL_RANK", "0")))     # same library instance
    try:
        return join_summary(bench_ops.bench_join(eng, 1.0, cases=((0.8, 0.15), (1.0, 1.0))), 1)
    except Exception as e:                                        # the headline line must survive
        return {"error": repr(e)}


def measure_ops(args):
    """The other BASELINE.json configs on one GPU, bounded: batched shared scan (config 2),
    index range select + fetch (config 3), hash join with prefilters (config 4); plus the two
    callers next to the path (SURVEY.md 8f): bulk CSV load and print of a long result."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_ops
    import analytical_database_b200 as adb
    eng = adb.Engine(int(os.environ.get("LOCAL_RANK", "0")))     # same library instance
    out = {}
    try:
        out["shared_scan_100q_100M"] = bench_ops.bench_shared(eng, 1.0)
        out["index_500M"] = bench_ops.bench_index(eng, 1.0)
        out["hash_join_100Mx100M"] = bench_ops.bench_join(eng, 1.0)
        out["csv_load_4M_rows"] = bench_ops.bench_load(eng, 1.0)          # SURVEY.md 8f rank 1
        out["print_50M_values"] = bench_ops.bench_print(eng, 1.0)         # SURVEY.md 8f rank 2
    except Exception as e:                                        # the headline line must survive
        out["error"] = repr(e)
    return out


def measure_cpu(args, eng, cols, res, shard_rows, lo, hi):
    """The reference's CPU operators on a bounded sample of the same table, on the box's
    host cores, checked against the GPU's result for the same rows."""
    ops, kind, what = cpu_ops()
    cores = os.cpu_count() or 1
    rows = min(args.cpu_rows, shard_rows)
    c1, c2 = cols[0]
    sel, fet = c1.to_host(rows), c2.to_host(rows)          # the very rows the GPU scanned
    (s1, h1) = ops.chain_select_fetch_sum(sel, fet, lo, hi, threads=1)
    t0 = time.perf_counter()
    ops.chain_select_fetch_sum(sel, fet, lo, hi, threads=1)
    t_single = time.perf_counter() - t0
    reps, t_all = 0, 0.0
    ops.chain_select_fetch_sum(sel, fet, lo, hi, threads=cores)
    t0 = time.perf_counter()
    while t_all < 8.0 and reps < 200:
        s2, h2 = ops.chain_select_fetch_sum(sel, fet, lo, hi, threads=cores)
        reps += 1
        t_all = time.perf_counter() - t0
    # parity: GPU chain on the same rows
    pos, val, cnt = res[0]
    h_cnt = C.c_int64(0)
    blo, bhi = C.c_int32(lo), C.c_int32(hi)
    eng._ck(eng.lib.adb_select_scan(c1.i32(), rows, C.byref(blo), C.byref(bhi), 0, pos.i32(),
                                    cnt.i64(), C.byref(h_cnt)))
    eng.fetch(c2, pos, h_cnt.value, out=val)
    g = eng.aggregate(val, h_cnt.value)
    ok = (g.sum, h_cnt.value) == (s1, h1) == (s2, h2)
    out = {"value": rows * reps / t_all, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": f"first {rows} rows of shard 0 (downloaded from HBM: identical rows), "
                     f"{reps} passes on {cores} threads (one reference instance per row range); {what}",
           "single_thread_value": rows / t_single, "parity_with_gpu": bool(ok)}
    from oracle import oracle
    r0 = oracle.reference("O0")
    if r0 is not None:
        t0 = time.perf_counter()
        r0.chain_select_fetch_sum(sel, fet, lo, hi, threads=1)
        out["single_thread_O0_value"] = rows / (time.perf_counter() - t0)
    if not ok:
        raise SystemExit(f"PARITY FAILURE: gpu {(g.sum, h_cnt.value)} cpu {(s1, h1)}")
    return out


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL's version banner, torchrun) write to fd 1; the contract is ONE JSON line
    on stdout.  Point fd 1 at stderr for the run and keep the real stdout for the result."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--selectivity", type=float, default=0.01)
    ap.add_argument("--cpu-rows", type=int, default=500_000_000,
                    help="rows of the cpu_baseline sample of the engine arm; the reference arm runs the "
                         "whole table unless --cpu-rows is given explicitly there (0 = whole table)")
    ap.add_argument("--shards-limit", type=int, default=0, help="debug: fewer shards per rank")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-cold", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-lazy", action="store_true", help="skip the unmaterialised (4N + 4H) chain")
    ap.add_argument("--no-configs", action="store_true",
                    help="skip BASELINE configs 2 (shared scan) and 3 (index) through the operator API")
    ap.add_argument("--no-join", action="store_true", help="skip the hash-join measurement (config 4)")
    ap.add_argument("--join-torch", action="store_true",
                    help="also time the process-per-GPU join of analytical-database_b200/sharded.py (peer exchange "
                         "vs NCCL all-to-all-v; round-1 form) and the single-GPU C-ABI join")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: aggregate exchange through the engine's peer-memory kernel or NCCL")
    ap.add_argument("--exchange-self", action="store_true",
                    help="debug (N = 1): run the last shard through the exchange-carrying chain kernel")
    ap.add_argument("--ops", action="store_true",
                    help="also time shared scan / index / join at the BASELINE config sizes")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="engine arm: after the timed steps, write what the chain computed in the last one "
                         "to DIR as .npy files (a seeded sample of every shard's lists; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "engine" else args.warmup
    quiet_stdout()
    if args.impl == "reference":
        if "--cpu-rows" not in sys.argv:
            args.cpu_rows = 0
        return run_reference(args)
    return run_engine(args)


if __name__ == "__main__":
    sys.exit(main())
