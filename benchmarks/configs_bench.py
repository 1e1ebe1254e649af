"""BASELINE.json configs 3, 4 and 5 as bench lines, sharded over N GPUs (one process per GPU, launched like bench.py):

    python bench.py --config 3 [--gpus N]     1e8 rows, 8 x Int64 with 10 % nulls: sum / min / max / count per column
    python bench.py --config 4 [--gpus N]     1e8 rows, Int32 -> Float64 cast, then xf + y, (xf + y) * y, sum
    python bench.py --config 5 [--gpus N]     Vec<RecordBatch> 256 x 4e6 rows, mixed Int64 / Float64, full pipeline

The Vec<RecordBatch> is split over the ranks by row range (configs 3, 4: parallel.shard_row_ranges) or by batch
(config 5: batch i -> rank i mod N); every rank generates ITS shard on the device with the counter-based generator
(the oracle regenerates any row), elementwise operators run without any exchange, and the aggregates come back
combined by the library's grouped ncclAllReduce.  Integer aggregates are checked against N = 1 values recorded in
tests/golden/configs_n1.json (identical for every N by construction); parity against the oracle at full size is
tests/test_configs_gpu.py (N = 1) and tests/comm_worker.py (N > 1).

Prints one JSON line (rank 0) in bench.py's format; `value` = rows of the table per second, whole job.
"""
from __future__ import annotations

import json
import os
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 20260924
CHUNK = 4_000_000
ROWS = 100_000_000

WORKLOADS = {
    3: "1e8 rows x 8 Int64 cols with 10% nulls (25 chunks x 4e6): sum/min/max/count per column, shard + NCCL combine",
    4: "1e8 rows: x Int32 (10% nulls) -> cast Float64, z = xf + y, w = z * y, s = sum(w)",
    5: "Vec<RecordBatch> 256 x 4e6 rows, i0,i1 Int64 + f0,f1 Float64 (5% nulls): f2=f0+f1; f3=f2*f0; i2=i0+i1; f4=cast(i2); f5=f3/f1; f6=sin(f5); f7=f6+f4; sum/min/max/count(i2), sum(f7), count(f7)",
}
METRICS = {3: "rows/s on 1e8-row 8xInt64 sum/min/max/count", 4: "rows/s on 1e8-row Int32->Float64 cast + arithmetic chain + sum",
           5: "rows/s on 256x4e6-row mixed Int64/Float64 scalar+aggregate pipeline"}


def _peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _my_rows(parallel, rank, world):
    """This rank's contiguous row range of the 25 x 4e6 table: (row0, chunk lengths)."""
    pieces = parallel.shard_row_ranges([CHUNK] * (ROWS // CHUNK), rank, world)
    lens = [n for _, _, n in pieces]
    row0 = pieces[0][0] * CHUNK + pieces[0][1] if pieces else 0
    return row0, lens


def _kernel_table(records, steps):
    by = {}
    for r in records:
        by.setdefault((r["kernel"], r["dtype"]), []).append(r)
    out = []
    peak, _ = _peak()
    for (k, dt), v in by.items():
        ms = float(np.mean([r["ms"] for r in v]))
        b = float(np.mean([r["bytes"] for r in v]))
        out.append({"kernel": k, "dtype": dt, "launches_per_step": len(v) / steps, "avg_ms": ms, "algorithmic_bytes": b,
                    "GBs": b / (ms * 1e-3) / 1e9 if ms else None, "frac_of_peak": b / (ms * 1e-3) / 1e9 / peak if ms else None})
    return out


def _time(ctx, step, steps, warmup, world, N):
    for _ in range(max(warmup, 2)):
        step()
    ctx.profile_read()
    ctx.profile_enable(True)
    ctx.comm_barrier()
    l0 = ctx.launch_count()
    ctx.timer_start()
    last = None
    for _ in range(steps):
        last = step()
    ms = ctx.timer_stop()
    ctx.comm_barrier()
    launches = ctx.launch_count() - l0
    ctx.profile_enable(False)
    recs = ctx.profile_read()
    if world > 1:
        ms = float(ctx.comm_all_reduce([ms], N.MAX)[0])
    return ms, last, launches, recs


def config3(rdf, N, parallel, ctx, rank, world, args):
    row0, lens = _my_rows(parallel, rank, world) if args.scaling == "strong" else (rank * ROWS, [CHUNK] * (ROWS // CHUNK))
    cols = [rdf.Column.generate(rdf.I64, lens, 2 if k == 7 else 3, col_id=30 + k, row0=row0, null_mod=10, ctx=ctx) for k in range(8)]
    ctx.synchronize()

    def step():
        return rdf.Column.aggregate_all_many(cols, asynchronous=True).result()   # 8 reductions, one host wait, ONE grouped collective

    ms, last, launches, recs = _time(ctx, step, args.steps, args.warmup, world, N)
    rows_total = ROWS * (world if args.scaling == "weak" else 1)
    check = {f"col{k}": {key: int(last[k][key]) for key in ("sum", "min", "max", "count", "rows")} for k in range(8)}
    bytes_per_step_rank = sum(lens) * 8 * 8.125
    return ms, rows_total, launches, recs, check, bytes_per_step_rank, cols


def config4(rdf, N, parallel, ctx, rank, world, args):
    row0, lens = _my_rows(parallel, rank, world) if args.scaling == "strong" else (rank * ROWS, [CHUNK] * (ROWS // CHUNK))
    x = rdf.Column.generate(rdf.I32, lens, 2, col_id=40, row0=row0, null_mod=10, ctx=ctx)
    y = rdf.Column.generate(rdf.F64, lens, 0, -1e3, 1e3, col_id=41, row0=row0, ctx=ctx)
    ctx.synchronize()

    def step():   # every intermediate is materialised as a column, like Evaluate::calculate does (src/evaluation.rs:66-96)
        xf = x.cast(rdf.F64)
        z = xf.add(y)
        w, fut = z.binary_agg_async(N.MUL, y)
        r = fut.result()
        for c in (xf, z, w):
            c.free()
        return r

    ms, last, launches, recs = _time(ctx, step, args.steps, args.warmup, world, N)
    rows_total = ROWS * (world if args.scaling == "weak" else 1)
    check = {"sum": float(last["sum"]), "count": int(last["count"]), "rows": int(last["rows"])}
    fused = None
    if not args.skip_e2e:   # the same chain through the fused-expression entry (cast folded into the load): 20 B/row instead of 60.75
        def step_fused():
            w, r = rdf.eval_expr_agg([x, y], [(N.ADD, 0, 1), (N.MUL, 2, 1)], materialise=True)
            w.free()
            return r

        fms, flast, _, _ = _time(ctx, step_fused, args.steps, args.warmup, world, N)
        fused = {"ms_per_step": fms / args.steps, "rows_per_s": rows_total * args.steps / (fms * 1e-3), "sum": float(flast["sum"]),
                 "bit_identical_sum": bool(np.float64(flast["sum"]).view(np.uint64) == np.float64(last["sum"]).view(np.uint64)) if world == 1 else None}
    bytes_per_step_rank = sum(lens) * (12.25 + 24.25 + 24.25)
    return ms, rows_total, launches, recs, check, bytes_per_step_rank, (x, y), fused


def main(args, rank, world, local):
    import rust_dataframe_b200 as rdf
    from rust_dataframe_b200 import native as N
    from rust_dataframe_b200 import parallel

    if args.impl == "reference":
        return reference_arm(args, rank)
    import bench

    bench.bind_to_gpu_numa_node(local)
    ctx = rdf.Context(local)
    if world > 1:
        parallel.attach_communicator(ctx)
    cfg = args.config
    extra = {}
    if cfg == 3:
        ms, rows_total, launches, recs, check, bytes_rank, keep = config3(rdf, N, parallel, ctx, rank, world, args)
    elif cfg == 4:
        ms, rows_total, launches, recs, check, bytes_rank, keep, fused = config4(rdf, N, parallel, ctx, rank, world, args)
        extra["fused_expression"] = fused
    else:
        ms, rows_total, launches, recs, check, bytes_rank, keep = config5_run(rdf, N, parallel, ctx, rank, world, args)
    if rank != 0:
        return
    peak, peak_src = _peak()
    table = _kernel_table(recs, args.steps)
    dom = max(table, key=lambda t: t["avg_ms"] * t["launches_per_step"]) if table else None
    golden = None
    gpath = os.path.join(ROOT, "tests", "golden", "configs_n1.json")
    if os.path.exists(gpath) and args.scaling == "strong":
        want = json.load(open(gpath)).get(str(cfg))
        if want is not None:
            if cfg == 3:
                golden = want == check
            elif cfg == 5:
                golden = all(want[k] == check[k] for k in want if k.startswith("i2_") or k.endswith("count"))
            else:
                golden = want["count"] == check["count"] and want["rows"] == check["rows"]
    line = {
        "metric": METRICS[cfg], "value": rows_total * args.steps / (ms * 1e-3), "unit": "rows/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 2), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "int64" if cfg == 3 else "f64", "data": "synthetic",
        "config": {"workload": WORKLOADS[cfg], "n_gpus": world, "scaling": args.scaling},
        "roofline": {"bound": "hbm", "kernel": dom and f'{dom["kernel"]} (dtype {dom["dtype"]})', "achieved": dom and dom["GBs"], "peak": peak, "unit": "GB/s",
                     "frac": dom and dom["frac_of_peak"], "traffic": None, "peak_source": peak_src,
                     "step_GBs_this_rank": bytes_rank / (ms / args.steps * 1e-3) / 1e9, "kernels": table},
        "gpu_launches": int(launches), "check": check, "matches_n1_golden": golden,
        "detail": {"collectives": ctx.comm_info()["collectives"], "nccl_version": ctx.comm_info()["nccl_version"]},
    }
    line.update(extra)
    print(json.dumps(line), flush=True)


def config5_run(rdf, N, parallel, ctx, rank, world, args):
    """Config 5 is 256 batches by definition (a strong series): rank r owns the contiguous block of 256/N batches that
    starts at batch r * 256/N (32 batches per GPU at N = 8) -- contiguous so that one generated column per input covers
    the shard (the generator numbers rows consecutively from row0); the batches are i.i.d., the block map balances exactly."""
    n_batches = 256
    per = n_batches // world
    assert per * world == n_batches, "config 5 needs the GPU count to divide 256"
    lens = [CHUNK] * per
    row0 = rank * per * CHUNK
    G = rdf.Column.generate
    i0 = G(rdf.I64, lens, 3, col_id=50, row0=row0, null_mod=20, ctx=ctx); i1 = G(rdf.I64, lens, 3, col_id=51, row0=row0, null_mod=20, ctx=ctx)
    f0 = G(rdf.F64, lens, 0, -1e3, 1e3, col_id=52, row0=row0, null_mod=20, ctx=ctx); f1 = G(rdf.F64, lens, 1, col_id=53, row0=row0, null_mod=20, ctx=ctx)
    ctx.synchronize()

    def step():
        f2 = f0.add(f1); f3 = f2.multiply(f0); f2.free()
        i2, fut_i2 = i0.binary_agg_async(N.ADD, i1)
        f4 = i2.cast(rdf.F64)
        f5 = f3.divide(f1); f3.free()
        f6 = f5.sin(); f5.free()
        f7, fut_f7 = f6.binary_agg_async(N.ADD, f4); f6.free()
        a, b = fut_i2.result(), fut_f7.result()
        for c in (i2, f4, f7):
            c.free()
        return a, b

    ms, last, launches, recs = _time(ctx, step, args.steps, min(args.warmup, 2), world, N)
    a, b = last
    check = {"i2_sum": int(a["sum"]), "i2_min": int(a["min"]), "i2_max": int(a["max"]), "i2_count": int(a["count"]), "f7_sum": float(b["sum"]),
             "f7_count": int(b["count"]), "rows": int(b["rows"])}
    bytes_rank = sum(lens) * (24.375 + 24.375 + 24.375 + 16.25 + 24.375 + 16.25 + 24.375)
    return ms, n_batches * CHUNK, launches, recs, check, bytes_rank, (i0, i1, f0, f1)


def reference_arm(args, rank):
    """The reference's CPU path for the config (oracle port), bounded sample: ONE chunk of 4e6 rows per column, scaled.
    A step is one pass of the config's operators over that chunk; --warmup untimed passes, then --steps timed ones."""
    if rank != 0:
        return
    from oracle import pyoracle as orc

    cfg = args.config
    if cfg == 3:
        cols = [[orc.generate(orc.I64, 2 if k == 7 else 3, 0, 0, SEED, 30 + k, 0, CHUNK, 10)] for k in range(8)]

        def step():
            for c in cols:   # sum, max, min are separate sequential passes; count is metadata (aggregate.rs:12-31,70-93)
                for op in (orc.SUM, orc.MAX, orc.MIN, orc.COUNT):
                    orc.aggregate(op, orc.I64, c)
    elif cfg == 4:
        x = [orc.generate(orc.I32, 2, 0, 0, SEED, 40, 0, CHUNK, 10)]
        y = [orc.generate(orc.F64, 0, -1e3, 1e3, SEED, 41, 0, CHUNK)]

        def step():
            _, xf = orc.col_cast(orc.I32, orc.F64, x)
            _, z = orc.col_binary(orc.ADD, orc.F64, xf, y)
            _, w = orc.col_binary(orc.MUL, orc.F64, z, y)
            orc.aggregate(orc.SUM, orc.F64, w)
    else:
        i0 = [orc.generate(orc.I64, 3, 0, 0, SEED, 50, 0, CHUNK, 20)]; i1 = [orc.generate(orc.I64, 3, 0, 0, SEED, 51, 0, CHUNK, 20)]
        f0 = [orc.generate(orc.F64, 0, -1e3, 1e3, SEED, 52, 0, CHUNK, 20)]; f1 = [orc.generate(orc.F64, 1, 0, 0, SEED, 53, 0, CHUNK, 20)]

        def step():
            _, f2 = orc.col_binary(orc.ADD, orc.F64, f0, f1); _, f3 = orc.col_binary(orc.MUL, orc.F64, f2, f0)
            _, i2 = orc.col_binary(orc.ADD, orc.I64, i0, i1); _, f4 = orc.col_cast(orc.I64, orc.F64, i2)
            _, f5 = orc.col_binary(orc.DIV, orc.F64, f3, f1); _, f6 = orc.col_unary(orc.SIN, orc.F64, f5)
            _, f7 = orc.col_binary(orc.ADD, orc.F64, f6, f4)
            for op in (orc.SUM, orc.MAX, orc.MIN, orc.COUNT):
                orc.aggregate(op, orc.I64, i2)
            orc.aggregate(orc.SUM, orc.F64, f7); orc.aggregate(orc.COUNT, orc.F64, f7)
    threads = 1
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = CHUNK * args.steps / dt
    line = {"impl": "reference", "metric": METRICS[cfg], "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "int64" if cfg == 3 else "f64",
            "data": "synthetic", "config": {"workload": WORKLOADS[cfg], "n_gpus": args.gpus, "scaling": args.scaling},
            "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port",
                             "sample": "ONE 4e6-row chunk per column through the oracle, sequential over chunks on one thread as the reference's subtract/multiply/divide/sin/sum/max are; rows/s of the chunk"},
            "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)
