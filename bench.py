#!/usr/bin/env python
"""bench.py -- rows/s on the 1e8-row f64 add+sum hot path (BASELINE.json `metric`), one process per GPU.

    python bench.py --gpus 1 --steps 50 --warmup 5              # this framework (CUDA, sm_100a)
    python bench.py --impl reference --gpus 1 --steps 5 ...     # the reference's CPU path (C restatement, host cores)
    torchrun --nproc-per-node N bench.py --gpus N ...           # N GPUs: weak series (1e8 rows per GPU) + strong series
    python bench.py --config 3|4|5 [--gpus N]                   # the other BASELINE configs (benchmarks/configs_bench.py)
    python bench.py ... --dump-outputs DIR                      # also write the last timed step's outputs as DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic input:
    c = ScalarFunctions::add(a, b)   (25 chunks x 4e6 rows of Float64, no nulls)   -> 24 B/row through HBM
    s = AggregateFunctions::sum(c)                                                  ->  8 B/row through HBM
`value` = rows/s with a and b already resident in HBM (c is materialised in HBM every step, s comes back to
the host every step).  At N > 1 every rank owns a shard of the Vec<RecordBatch>; the per-GPU partial sums are
combined by the LIBRARY with one grouped ncclAllReduce per step, enqueued on the stream that produced them
(csrc/comm.cu) -- bench.py itself issues no collective inside the timed loop.
`e2e`   = the same two operators through the drop-in host entries the Rust shim binds (bdf_binary + bdf_aggregate)
with HOST buffers (pinned once, outside the loop): a and b are copied to the device inside the timed region, c is copied
back to host memory, then sum(c) reads the host copy of c again (two calls, as the reference API is two calls).
`e2e.variants` holds the same sequence on pageable buffers (fresh / reused outputs) and the device-column chain.
Prints exactly one JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROWS = 100_000_000
CHUNK = 4_000_000
SEED = 20260924
METRIC = "rows/s on 1e8-row f64 add+sum"
WORKLOAD = "1e8 rows x 2 Float64 cols (25 chunks x 4e6 rows, no nulls): c = a + b, then sum(c)"


def config_dict(n_gpus: int, scaling: str) -> dict:
    """Identical in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "rows": ROWS, "chunks": ROWS // CHUNK, "chunk_rows": CHUNK, "n_gpus": n_gpus, "scaling": scaling,
            "rows_are": "per GPU (weak)" if scaling == "weak" else "in total, split over the GPUs by row range (strong)"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _nvml_index(cuda_index: int) -> int:
    """CUDA ordinal -> NVML index when CUDA_VISIBLE_DEVICES is a plain list of integers (otherwise the ordinal itself)."""
    cvd = os.environ.get("CUDA_VISIBLE_DEVICES", "")
    try:
        ids = [int(x) for x in cvd.split(",") if x.strip() != ""]
        return ids[cuda_index] if cuda_index < len(ids) else cuda_index
    except ValueError:
        return cuda_index


class ClockSampler(threading.Thread):
    """Polls NVML for SM clock and throttle reasons while the timed region runs.  ONE poller per job: rank 0 watches every GPU of
    the job (eight processes polling NVML at once starved each other: one sample in 140 ms at N = 8); the other ranks pass []."""

    def __init__(self, device_indices):
        super().__init__(daemon=True)
        self.samples = []          # (time, [mhz per GPU], OR of the reasons)
        self.stop_flag = False
        self.ok = False
        self.err = "not polled on this rank (rank 0 watches every GPU of the job)"
        self.handles = []
        if not device_indices:
            return
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            for d in device_indices:
                self.handles.append(pynvml.nvmlDeviceGetHandleByIndex(_nvml_index(int(d))))
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handles[0], pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = str(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz, reasons = [], 0
                for h in self.handles:
                    mhz.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    reasons |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                self.samples.append((time.perf_counter(), mhz, reasons))
            except Exception:
                pass
            time.sleep(0.01)   # ~15 samples over the 150 ms window; a tighter loop would compete with rank 0's hot loop for the GIL

    def summary(self, t0: float, t1: float):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + str(self.err)]}
        nv = self.nv
        win = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-3:]
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        seen = set()
        for _, _, r in win:
            for bit, name in names.items():
                if r & bit:
                    seen.add(name)
        every = [m for s in win for m in s[1]]
        out = {"sm_mhz": float(np.median(every)) if every else None, "sm_max_mhz": float(self.max_mhz),
               "reasons": sorted(seen), "samples": len(win), "gpus_watched": len(self.handles)}
        if len(self.handles) > 1 and win:
            out["sm_mhz_per_gpu"] = [float(np.median([s[1][g] for s in win])) for g in range(len(self.handles))]
        return out


def bind_to_gpu_numa_node(device_index: int):
    """Pin this process (and therefore its pinned host buffers, by first touch) to the NUMA node the GPU hangs off.
    Pure placement: host<->device copies then do not cross the inter-socket link.  Best effort."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        path = f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def env_ranks():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


DUMP_ROWS = 1 << 22   # rows of c that --dump-outputs writes: 32 MB of float64


def dump_rows(n: int) -> np.ndarray:
    """The row numbers of c that --dump-outputs writes, for a c of n rows: drawn with a fixed seed, the same on every run."""
    return np.sort(np.random.default_rng(SEED).integers(0, n, min(DUMP_ROWS, n)))


def dump_outputs(out_dir: str, c_chunks, s: float, count: int):
    """--dump-outputs: what the last timed step returned to its caller, so that two builds can be compared output for output.
    c.npy holds the values of c at the rows dump_rows picks (c has no nulls in this workload, so it carries no validity),
    sum.npy holds sum(c) and count.npy the number of rows it counted.  At N > 1 rank 0 writes what its caller receives:
    its own shard of c beside the sum and count combined over every rank."""
    c = np.concatenate(c_chunks)
    rows = dump_rows(c.shape[0])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "c.npy"), c[rows])
    np.save(os.path.join(out_dir, "sum.npy"), np.array([s], np.float64))
    np.save(os.path.join(out_dir, "count.npy"), np.array([count], np.float64))


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the reference's CPU path (C restatement in oracle/, see oracle/oracle.h for provenance)

def cpu_step_factory(rows: int):
    from oracle import pyoracle as orc

    n_chunks = max(1, rows // CHUNK)
    lens = [CHUNK] * n_chunks
    a = [orc.generate(orc.F64, 0, -1e3, 1e3, SEED, 0, i * CHUNK, n) for i, n in enumerate(lens)]
    b = [orc.generate(orc.F64, 0, -1e3, 1e3, SEED, 1, i * CHUNK, n) for i, n in enumerate(lens)]
    threads = max(1, min(os.cpu_count() or 1, n_chunks))
    views_a, views_b = orc._views(a), orc._views(b)
    outs, bufs = orc._alloc_outs(orc.F64, lens)  # output buffers allocated once (arrow allocates per call)
    L = orc.lib()
    import ctypes as C

    res = np.zeros(1)
    some = C.c_int32(0)
    out_views = (orc.View * n_chunks)()
    for i, (v, _) in enumerate(bufs):
        out_views[i].values = v.ctypes.data
        out_views[i].validity = None
        out_views[i].len = lens[i]
        out_views[i].offset = 0
        out_views[i].null_count = 0

    def step():
        # ScalarFunctions::add: rayon par_iter over chunks (scalar.rs:28-31) -> one thread per chunk up to nproc
        st = L.orc_col_binary(orc.ADD, orc.F64, n_chunks, views_a, n_chunks, views_b, outs, threads)
        assert st == 0
        # AggregateFunctions::sum: chunks in order on the calling thread, sequential fold (aggregate.rs:82-93)
        st = L.orc_aggregate(orc.SUM, orc.F64, n_chunks, out_views, res.ctypes.data, C.byref(some))
        assert st == 0
        return float(res[0])

    step._keep = (a, b, bufs, views_a, views_b, outs, out_views)  # the ctypes views hold raw pointers into these
    return step, n_chunks * CHUNK, threads


REF_NOTE = ("CPU path of the reference: C restatement of rust-dataframe @ a8310afd + arrow-rs~2.0 semantics (oracle/oracle.c); "
            "the Rust reference cannot be built in this image")


def run_reference_arm(args, rank: int, world: int):
    if rank != 0:
        return
    step, rows, threads = cpu_step_factory(ROWS)   # always the full workload: the sample never shrinks silently
    assert rows == ROWS
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        s = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs is not None:
        _, _, bufs, _, _, outs, _ = step._keep
        dump_outputs(args.dump_outputs, [v for v, _ in bufs], s, sum(len(v) - outs[i].null_count for i, (v, _) in enumerate(bufs)))
    value = rows * args.steps / dt
    sample = (f"{rows} rows ({rows // CHUNK} chunks x {CHUNK}) per step, {args.steps} steps; add on {threads} threads (one per chunk, rayon mirror), "
              f"sum on 1 thread; output buffers allocated once")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(args.gpus, args.scaling),
        "detail": {"note": REF_NOTE, "rows_per_step": rows, "host_cpus": os.cpu_count()},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# GPU arm

def make_inputs(rdf, ctx, rank: int, world: int, scaling: str):
    """This rank's shard of the two input columns, generated on the device (counter-based generator: the oracle can
    regenerate any row).  weak: 25 x 4e6 rows per rank; strong: the same 1e8 rows split by row range."""
    from rust_dataframe_b200 import parallel

    if scaling == "weak":
        lens = [CHUNK] * (ROWS // CHUNK)
        row0 = rank * ROWS
        pieces = [(row0 + i * CHUNK, CHUNK) for i in range(len(lens))]
    else:
        full = [CHUNK] * (ROWS // CHUNK)
        pieces = [(i * CHUNK + start, n) for i, start, n in parallel.shard_row_ranges(full, rank, world)]
    # consecutive pieces form one generated column (row0 of piece k+1 = row0 of piece k + its length: contiguous ranges)
    lens = [n for _, n in pieces]
    row0 = pieces[0][0] if pieces else 0
    a = rdf.Column.generate(rdf.F64, lens, 0, -1e3, 1e3, seed=SEED, col_id=0, row0=row0, ctx=ctx)
    b = rdf.Column.generate(rdf.F64, lens, 0, -1e3, 1e3, seed=SEED, col_id=1, row0=row0, ctx=ctx)
    ctx.synchronize()
    return a, b, lens


class HotLoop:
    """c = a + b materialised in HBM with sum(c) folded into the same pass (K5); the host keeps `depth` steps in flight:
    step i's scalar (already combined across the ranks by the library) is fetched after step i+depth is enqueued."""

    def __init__(self, N, a, b, depth: int):
        self.N, self.a, self.b, self.depth = N, a, b, depth
        self.inflight = []
        self.last = None
        self.last_c = None

    def retire(self, keep: bool = False):
        c, fut = self.inflight.pop(0)
        r = fut.result()
        if keep:
            self.last_c = c
        else:
            c.free()
        self.last = (float(r["sum"]), int(r["count"]), int(r["rows"]))

    def step(self):
        self.inflight.append(self.a.binary_agg_async(self.N.ADD, self.b))
        if len(self.inflight) > self.depth:
            self.retire()

    def drain(self, keep_last: bool = False):
        """keep_last: the last step's c is left allocated in last_c (for --dump-outputs) instead of freed."""
        while self.inflight:
            self.retire(keep=keep_last and len(self.inflight) == 1)
        return self.last


def timed_loop(ctx, loop: HotLoop, steps: int, world: int, keep_last: bool = False):
    """barrier; K steps between two events on the compute stream; drain; barrier.  Returns max-over-ranks ms."""
    ctx.comm_barrier()
    ctx.timer_start()
    for _ in range(steps):
        loop.step()
    loop.drain(keep_last)
    ms = ctx.timer_stop()
    ctx.comm_barrier()
    if world > 1:
        from rust_dataframe_b200 import native as N

        ms = float(ctx.comm_all_reduce([ms], N.MAX)[0])
    return ms


def run_gpu_arm(args, rank: int, world: int, local: int):
    import rust_dataframe_b200 as rdf
    from rust_dataframe_b200 import native as N
    from rust_dataframe_b200 import parallel

    ctx = rdf.Context(local)
    if world > 1:
        parallel.attach_communicator(ctx)   # ncclCommInitRank inside libb200df; aggregates are collective from here on
    depth = 1 if world == 1 else int(os.environ.get("BDF_BENCH_DEPTH", "3"))
    warmup = max(args.warmup, 3)

    a, b, lens = make_inputs(rdf, ctx, rank, world, args.scaling)
    rows_local = sum(lens)
    rows_global = ROWS * world if args.scaling == "weak" else ROWS
    loop = HotLoop(N, a, b, depth)
    for _ in range(warmup):
        loop.step()
    loop.drain()

    # secondary figure: the unfused, blocking two-call sequence (what a caller of add() then sum() gets on device columns)
    def step_two_call():
        c = a.add(b)
        s = c.sum()          # collective at N > 1: the library returns the global sum
        c.free()
        return float(s)

    two_steps = max(3, min(args.steps, 20))
    for _ in range(3):
        step_two_call()
    ctx.comm_barrier()
    ctx.timer_start()
    for _ in range(two_steps):
        step_two_call()
    two_call_ms = ctx.timer_stop() / two_steps

    # cost of the combine alone: a blocking 4-in-1 aggregate of a tiny column with the collective on and off
    combine_us = None
    primary_mode = ctx.comm_get_combine() if world > 1 else None
    if world > 1:
        tiny = rdf.Column.generate(rdf.I64, [1024], 3, seed=SEED, col_id=9, row0=rank * 1024, ctx=ctx)
        reps = 200

        def blocking_us(collective: bool):
            ctx.comm_collective(collective)
            for _ in range(20):
                tiny.aggregate_all_async().result()
            ctx.comm_barrier() if collective else ctx.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                tiny.aggregate_all_async().result()
            return (time.perf_counter() - t0) / reps * 1e6

        local_us = blocking_us(False)
        combine_us = {"blocking_aggregate_local_us": local_us}
        modes = [primary_mode]
        try:   # the other transport, if the box offers it
            ctx.comm_set_combine(primary_mode != "peer-memory")
            modes.append(ctx.comm_get_combine())
            ctx.comm_set_combine(primary_mode == "peer-memory")
        except rdf.ArrowError:
            pass
        for m in modes:
            ctx.comm_set_combine(m == "peer-memory")
            us = blocking_us(True)
            combine_us[m] = {"blocking_aggregate_collective_us": us, "combine_us": us - local_us}
        ctx.comm_set_combine(primary_mode == "peer-memory")
        ctx.comm_collective(True)
        tiny.free()

    sampler = ClockSampler(list(range(world)) if rank == 0 else [])   # one node: the job's GPUs are local ranks 0..world-1
    sampler.start()
    ctx.profile_read()  # drop warm-up records
    ctx.profile_enable(True)
    launches0 = ctx.launch_count()
    coll0 = ctx.comm_info()["collectives"]
    t_wall0 = time.perf_counter()
    ms = timed_loop(ctx, loop, args.steps, world, keep_last=args.dump_outputs is not None)
    t_wall1 = time.perf_counter()
    launches = ctx.launch_count() - launches0
    collectives = ctx.comm_info()["collectives"] - coll0
    ctx.profile_enable(False)
    records = ctx.profile_read()
    last = loop.last
    # The timed window of the default run is a few ms: keep the same load running, untimed, for a FIXED number of extra steps
    # (derived from the max-over-ranks time, so every rank runs the same count -- each step enqueues a collective) so that
    # the NVML poller sees the clocks under this load.
    extra = int(min(5000, max(0, math.ceil(150.0 / max(ms / args.steps, 1e-3)) - args.steps)))
    for _ in range(extra):
        loop.step()
    loop.drain()
    ctx.comm_barrier()
    t_wall2 = time.perf_counter()
    sampler.stop_flag = True
    sampler.join(timeout=1)
    clocks = sampler.summary(t_wall0, t_wall2)
    clocks["window"] = f"timed region + {extra} untimed steps of the same load"
    if loop.last_c is not None:
        if rank == 0:   # at N > 1, c is rank 0's shard and the sum is the combined one
            dump_outputs(args.dump_outputs, [x.value_slice() for x in loop.last_c.download()], last[0], last[1])
        loop.last_c.free()
        loop.last_c = None

    # ---- the same series with the other transport of the combine (N > 1) ----
    other_transport = None
    if world > 1 and combine_us is not None and len(combine_us) > 2:
        alt = [m for m in combine_us if m not in ("blocking_aggregate_local_us", primary_mode)][0]
        ctx.comm_set_combine(alt == "peer-memory")
        for _ in range(3):
            loop.step()
        loop.drain()
        ms_alt = timed_loop(ctx, loop, args.steps, world)
        ctx.comm_set_combine(primary_mode == "peer-memory")
        other_transport = {"combine": alt, "value": rows_global * args.steps / (ms_alt * 1e-3), "ms_per_step": ms_alt / args.steps}

    # ---- the other scaling series (N > 1): same loop over the other sharding ----
    other = None
    if world > 1 and not args.skip_other_series:
        other_mode = "strong" if args.scaling == "weak" else "weak"
        a.free(); b.free()
        a, b, lens2 = make_inputs(rdf, ctx, rank, world, other_mode)
        loop2 = HotLoop(N, a, b, depth)
        for _ in range(warmup):
            loop2.step()
        loop2.drain()
        ms2 = timed_loop(ctx, loop2, args.steps, world)
        rows2 = ROWS * world if other_mode == "weak" else ROWS
        other = {"scaling": other_mode, "value": rows2 * args.steps / (ms2 * 1e-3), "unit": "rows/s", "ms_per_step": ms2 / args.steps,
                 "rows_total": rows2, "rows_this_rank": sum(lens2), "check": {"sum": loop2.last[0], "count": loop2.last[1]}}
        a.free(); b.free()
        a, b, lens = make_inputs(rdf, ctx, rank, world, args.scaling)

    # ---- e2e: host buffers, copies inside the timed region ----
    e2e = None if args.skip_e2e else run_e2e(args, ctx, rdf, N, lens, a, b, world, local)

    if rank != 0:
        return
    peak, peak_src = measured_peaks()
    bins = [r for r in records if r["kernel"] == "binary"]
    add_ms = float(np.mean([r["ms"] for r in bins])) if bins else None
    add_bytes = bins[0]["bytes"] if bins else 24 * rows_local
    achieved = add_bytes / (add_ms * 1e-3) / 1e9 if add_ms else None
    roofline = {
        "bound": "hbm", "kernel": "k_binary<double,ADD,AGG> (one launch over this rank's chunks)", "achieved": achieved, "peak": peak,
        "unit": "GB/s", "frac": achieved / peak if achieved else None, "traffic": None,
        "traffic_source": None, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": add_bytes, "avg_launch_ms": add_ms, "frac_of_8TBs_nominal": achieved / 8000.0 if achieved else None,
        "step_GBs_algorithmic_24B_per_row": 24 * rows_local / (ms / args.steps * 1e-3) / 1e9,
        "two_call_unfused": {"ms_per_step": two_call_ms, "rows_per_s": rows_global / (two_call_ms * 1e-3),
                             "note": "blocking add() then sum() on device columns: 32 B/row, two kernels + a host sync (+ the combine) per step"},
    }
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file) and args.scaling == "weak":
        with open(traffic_file) as f:
            tj = json.load(f)
        roofline["traffic"] = tj.get("k_binary_f64_add_bytes_per_launch")
        roofline["traffic_source"] = "static: ncu --set full capture committed under profiles/ (%s), not re-measured by this run" % tj.get("source", "profiles/traffic.json")

    cpu = None if args.skip_cpu else run_cpu_baseline()

    value = rows_global * args.steps / (ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_dict(world, args.scaling),
        "detail": {"rows_this_rank": rows_local, "chunks_this_rank": len(lens), "parallelism": f"shard{world}",
                   "l2": "inputs (2.4 GB working set per step at 1e8 rows) are larger than the 126 MB L2; no flush needed",
                   "fused": "sum(c) is computed by the add kernel while c is written (c is still materialised): 24 B/row",
                   "host_pipelining": f"{depth} step(s) in flight: step i's scalar is read after step i+{depth} is enqueued",
                   "collective": "none" if world == 1 else "ONE combine of the partial (sum,count,rows,min,max) per step, enqueued by libb200df on the stream that produced it -- NVLink peer-memory mailboxes (k_p2p_combine) or the grouped ncclAllReduce, see combine_transport; no collective is issued by bench.py inside the timed loop",
                   "collectives_in_timed_region": int(collectives), "nccl_version": ctx.comm_info()["nccl_version"],
                   "combine_transport": primary_mode, "combine": combine_us, "same_series_other_transport": other_transport},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "check": {"sum": last[0], "count": last[1], "rows": last[2]},
    }
    if other is not None:
        line["other_series"] = other
    print(json.dumps(line), flush=True)


def run_e2e(args, ctx, rdf, N, lens, dev_a, dev_b, world, local):
    """The drop-in host entries with HOST buffers, H2D + D2H inside the timed region.  Variants:
      dropin_pageable_fresh   a, b pageable; c into freshly allocated pageable buffers every step (MutableBuffer::new)
      dropin_pageable_reused  a, b pageable; c into the same pageable buffers every step (an allocator that recycles)
      dropin_registered       a, b and c in memory pinned once outside the loop (bdf_host_alloc / bdf_host_register)
      device_chain_pinned     upload_many -> add with the sum folded in -> download (one PCIe crossing of c, pinned)
    Each drop-in step = ScalarFunctions.add(a, b) [bdf_binary] then AggregateFunctions.sum(c) [bdf_aggregate]."""
    steps = max(3, min(args.steps, 6))
    n_rows = sum(lens)
    # host copies of the same synthetic columns
    pin_a = N.alloc_outputs(rdf.F64, lens, ctx, pinned=True)
    pin_b = N.alloc_outputs(rdf.F64, lens, ctx, pinned=True)
    host_a_pin = dev_a.download(into=pin_a)
    host_b_pin = dev_b.download(into=pin_b)
    host_a = [rdf.PrimitiveArray.from_numpy(x.value_slice().copy()) for x in host_a_pin]   # plain malloc'ed memory
    host_b = [rdf.PrimitiveArray.from_numpy(x.value_slice().copy()) for x in host_b_pin]
    pin_out = N.alloc_outputs(rdf.F64, lens, ctx, pinned=True)
    reuse_out = N.alloc_outputs(rdf.F64, lens, ctx, pinned=False)
    for v, _, _ in reuse_out[1]:
        v[:] = 0.0  # fault the pages in once

    def dropin(a, b, into):
        outs, bufs = into if into is not None else N.alloc_outputs(rdf.F64, lens, ctx, pinned=False)
        for i in range(len(bufs)):
            outs[i].len = bufs[i][0].shape[0]
        N.raise_for_status(N.lib().bdf_binary(ctx.handle, N.ADD, rdf.F64, len(a), N.make_views(a), len(b), N.make_views(b), outs))
        c = N.collect_outputs(rdf.F64, outs, bufs)
        return float(rdf.AggregateFunctions.sum(c, dtype=rdf.F64, ctx=ctx))

    def chain():
        ca, cb = rdf.Column.upload_many([host_a_pin, host_b_pin], ctx=ctx, asynchronous=True)  # a0,b0,a1,b1,... over PCIe
        cc, fut = ca.binary_agg_async(N.ADD, cb)      # per upload group, as soon as its chunks have landed
        cc.download_begin(pin_out)                    # D2H of group g overlaps H2D of group g+1
        r = fut.result()
        cc.download_end(pin_out)
        for col in (ca, cb, cc):
            col.free()
        return float(r["sum"])

    variants = {
        "dropin_pageable_fresh": (lambda: dropin(host_a, host_b, None), 3 * 8 * n_rows, 8 * n_rows + 8),
        "dropin_pageable_reused": (lambda: dropin(host_a, host_b, reuse_out), 3 * 8 * n_rows, 8 * n_rows + 8),
        "dropin_registered": (lambda: dropin(host_a_pin, host_b_pin, pin_out), 3 * 8 * n_rows, 8 * n_rows + 8),
        "device_chain_pinned": (chain, 2 * 8 * n_rows, 8 * n_rows + 8),
    }
    out = {}
    for name, (fn, h2d, d2h) in variants.items():
        for _ in range(2):
            fn()
        ctx.comm_barrier()
        t0 = time.perf_counter()
        last = None
        for _ in range(steps):
            last = fn()
        ctx.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        ctx.comm_barrier()
        if world > 1:
            ms = float(ctx.comm_all_reduce([ms], N.MAX)[0])
        rows_total = ROWS * world if args.scaling == "weak" else ROWS
        out[name] = {"value": rows_total * steps / (ms * 1e-3), "unit": "rows/s", "ms_per_step": ms / steps, "h2d_bytes_per_step": h2d,
                     "d2h_bytes_per_step": d2h, "pcie_GBs_this_rank": (h2d + d2h) / (ms / steps * 1e-3) / 1e9, "check_sum": last}
    # Headline: the drop-in entries on host buffers that were pinned ONCE (bdf_host_register / bdf_host_alloc outside the loop) --
    # the memory mode BASELINE.json's north_star prescribes ("Arrow column data + validity buffers are pinned and copied to
    # device once per batch").  The pageable variants are reported beside it: they stage every byte through pinned slots
    # (a second pass over host DRAM), which one GPU sustains at ~45 GB/s but which does not scale past ~2 GPUs per socket.
    head = dict(out["dropin_registered"])
    head.update({"steps": steps, "timer": "host wall clock around the blocking calls (they return when the results are in host memory), max over ranks",
                 "api": "ScalarFunctions.add(a, b) -> bdf_binary(ADD), c written to host buffers; then AggregateFunctions.sum(c) -> bdf_aggregate(SUM) "
                        "re-reading c from the host (two calls, like the reference API); a, b and c live in host memory pinned once outside the loop",
                 "variants": {k: v for k, v in out.items() if k != "dropin_registered"}})
    return head


def run_cpu_baseline():
    """Oracle ('port' of the reference's CPU path) timed on this box's host cores, bounded sample."""
    try:
        step, rows, threads = cpu_step_factory(ROWS)
        step()
        reps, t0 = 0, time.perf_counter()
        while reps < 3 or (time.perf_counter() - t0 < 8 and reps < 40):
            step()
            reps += 1
        dt = time.perf_counter() - t0
        res_pa = None
        try:  # secondary reference point, NOT the reference: Arrow C++ via pyarrow on the same workload
            import pyarrow as pa
            import pyarrow.compute as pc

            a_np, b_np, _, _, _, _, _ = step._keep
            ca = pa.chunked_array([pa.array(x.values) for x in a_np])
            cb = pa.chunked_array([pa.array(x.values) for x in b_np])
            pc.sum(pc.add(ca, cb))
            t1 = time.perf_counter()
            pc.sum(pc.add(ca, cb))
            res_pa = {"rows_per_s": rows / (time.perf_counter() - t1), "note": "pyarrow %s pc.add + pc.sum (Arrow C++, differs from arrow-rs on f64 div-by-zero, casts, sum order)" % pa.__version__}
        except Exception as e:  # pragma: no cover
            res_pa = {"rows_per_s": None, "note": f"unavailable: {e}"}
        return {"value": rows * reps / dt, "unit": "rows/s", "cores": threads, "kind": "port", "arrow_cpp_pyarrow": res_pa,
                "sample": f"{reps} passes over the full {rows}-row workload; add on {threads} threads (one per chunk, like rayon), sum sequential on 1 thread; output buffers allocated once; host has {os.cpu_count()} cpus",
                "ms_per_step": dt / reps * 1e3}
    except Exception as e:  # pragma: no cover
        return {"value": None, "unit": "rows/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}


def _positive_int(s: str) -> int:
    n = int(s)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {n}")
    return n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive_int, default=100, help="timed steps")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="primary series (default: weak for the headline metric, strong for configs 3/4/5); at N > 1 the headline run measures the other one too and reports it under other_series")
    ap.add_argument("--config", type=int, default=1, choices=[1, 3, 4, 5], help="1 = the headline metric; 3/4/5 = the other BASELINE configs")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap.add_argument("--skip-cpu", action="store_true", help="profiling runs only: skip the CPU baseline leg")
    ap.add_argument("--skip-other-series", action="store_true", help="N > 1: measure only the primary scaling series")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/{c,sum,count}.npy (c: a fixed, seeded sample of rows)")
    args = ap.parse_args()
    if args.dump_outputs is not None and args.config != 1:
        ap.error("--dump-outputs applies to the headline workload (--config 1)")
    if args.scaling is None:
        args.scaling = "weak" if args.config == 1 else "strong"
    rank, world, local = env_ranks()
    if args.config != 1:
        from benchmarks import configs_bench

        configs_bench.main(args, rank, world, local)
        return
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    bind_to_gpu_numa_node(local)
    run_gpu_arm(args, rank, world, local)


if __name__ == "__main__":
    main()
