#!/usr/bin/env python
"""Benchmark of the hot path: TPC-H Q1/Q6/Q3 pipelines on TPC-H-shaped synthetic data.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--sf SF] [--impl ours|reference] [--dump-outputs DIR]

Metric (BASELINE.json): lineitem tuples/s over Q1+Q6+Q3 at SF100 (+ fraction of the HBM roofline).
A step = one pass of the three queries over the resident tables (3 scans of lineitem plus the
orders/customer build pipelines of Q3). `value` is timed with the tables resident in HBM;
`e2e` re-uploads the tables from pinned host memory through the C ABI every step.
N > 1: one process per GPU (torchrun), lineitem row-range sharded, SF fixed (strong scaling),
partial aggregates merged inside the library with NCCL.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

BYTES_PER_TUPLE = {"q1": 38, "q6": 28, "q3": 24}     # SURVEY.md 8(d): widths of the touched lineitem columns
QUERIES = ("q1", "q6", "q3")


def load_plan(name):
    with open(os.path.join(ROOT, "tests/golden/plans", name + ".json")) as f:
        return json.load(f)


def dump_outputs(out_dir, results, max_bytes=64 << 20):
    """Writes the result columns a caller of rq_plan_execute received, one `<query>.<column>.npy` per
    column, so that two builds can be compared output for output on the same seeded inputs. Integer
    columns (DECIMAL as scaled integers) become float64, strings a (rows, width) float32 array of their
    bytes. A result larger than its share of `max_bytes` is reduced to a fixed, seeded sample of rows,
    the same rows in every column, whose indices go to `<query>.rows.npy`."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for q, res in results.items():
        names = res.names or [f"col{i}" for i in range(len(res.columns))]
        row_bytes = 8 + sum(8 if c.dtype.kind != "S" else 4 * c.dtype.itemsize for c in res.columns)
        keep = (max_bytes // len(results)) // row_bytes
        rows = None
        if res.n_rows > keep:
            rows = np.sort(np.random.default_rng(0).choice(res.n_rows, size=keep, replace=False))
            np.save(os.path.join(out_dir, f"{q}.rows.npy"), rows.astype(np.float64))
        for i, (name, col) in enumerate(zip(names, res.columns)):
            if rows is not None:
                col = col[rows]
            if col.dtype.kind == "S":
                arr = col.view(np.uint8).reshape(len(col), col.dtype.itemsize).astype(np.float32)
            else:
                arr = col.astype(np.float64)
            np.save(os.path.join(out_dir, f"{q}.{i:02d}_{name}.npy"), arr)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                d = json.load(f)
            for key in ("hbm_gbs", "hbm_gbs_burst", "hbm_gbs_sustained"):
                if key in d and float(d[key]) > 0:
                    return float(d[key]), f"measured (MEASURED_PEAKS.json {key})"
        except (OSError, ValueError, TypeError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region"""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.stop = False
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i] == "Active" for s in self.samples)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(self.samples[0][1]),
                "reasons": reasons, "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference engine itself (oracle/_ref/resql-oracle)
# ---------------------------------------------------------------------------------------------
def run_reference(sample_sf, reps, threads):
    """Times the UNMODIFIED reference (its own JIT, `threads=<all cores>`) on a bounded sample of
    the same workload. Returns dict with tuples/s and per-query execute ms."""
    from resql_b200 import tpch
    from golden.queries import QUERIES as SQL
    exe = os.path.join(ROOT, "oracle/_ref/resql-oracle")
    kind = "reference"
    if not os.path.exists(exe):
        return None
    data = tpch.generate(sample_sf, seed=42, tables=("lineitem", "orders", "customer"))
    n = len(data["lineitem"]["l_orderkey"])
    with tempfile.TemporaryDirectory() as tmp:
        create = os.path.join(tmp, "create.sql")
        stm = []
        for name in ("lineitem", "orders", "customer"):
            fields = []
            for c, k, a in tpch.SCHEMAS[name]:
                ty = {"int": "int", "date": "date"}.get(k) or (f"decimal(12,{a})" if k == "dec" else f"{k}({a})")
                fields.append(f"{c} {ty}")
            stm.append(f"create table {name} ( " + ", ".join(fields) + " )")
        with open(create, "w") as f:
            f.write(";\n".join(stm) + ";\n")
        args = [exe, "--quiet", f"exec {create}"]
        for name in ("lineitem", "orders", "customer"):
            p = os.path.join(tmp, name + ".bin")
            tpch.to_rows(name, data[name]).tofile(p)
            del data[name]
            args.append(f"binload {name} {p}")
        args += [f"threads={threads}", f"repeat {reps}"]
        for q in QUERIES:
            args.append(" ".join(SQL[q].split()))
        t0 = time.perf_counter()
        r = subprocess.run(args, capture_output=True, text=True, timeout=1500)
        wall = time.perf_counter() - t0
    ms = [float(l.split("execute_ms=")[1]) for l in r.stdout.split("\n") if l.startswith("#select")]
    if len(ms) != reps * len(QUERIES):
        raise RuntimeError("reference run failed: " + r.stdout[-400:] + r.stderr[-400:])
    per_q = {q: ms[i * reps:(i + 1) * reps] for i, q in enumerate(QUERIES)}
    return {"kind": kind, "rows": n, "per_query_ms": per_q, "wall_s": wall, "threads": threads}


def run_reference_with_fallback(a, reps, threads):
    """the CPU sample at --sample-sf; if that does not fit the box (temporary files, memory), at SF1"""
    try:
        return run_reference(a.sample_sf, reps, threads)
    except Exception as e:      # noqa: BLE001
        if a.sample_sf <= 1.0:
            raise
        print(f"bench.py: CPU sample at SF{a.sample_sf:g} failed ({e}); falling back to SF1", file=sys.stderr)
        a.sample_sf = 1.0
        return run_reference(1.0, reps, threads)


# ---------------------------------------------------------------------------------------------
# --workload micro: the reference's README microbenchmark (README:69, BASELINE config 5)
#     select c, avg(d * a) from foo, bar where a = d group by c order by c
# foo(a, c) and bar(d) have N rows each; a and d are permutations of 1..N (every foo row joins exactly
# one bar row), c has G distinct values. With more than one GPU BOTH tables are row-range sharded and
# the plan runs with RQ_PLAN_PARTITIONED: build and probe rows are shipped to the rank that owns
# hash(key) (grouped ncclSend/ncclRecv), joined there, the partial groups are merged on the rank that
# owns hash(c), the result is concatenated and ordered. Every result is compared with an independent
# torch int64 evaluation (d * a = a * a because of the permutation property; wrap-around sums,
# truncating AVG), all-reduced over the ranks. One JSON line per case.
# ---------------------------------------------------------------------------------------------
def main_micro(a):
    import torch
    import torch.distributed as dist
    from resql_b200 import Engine, Plan
    from resql_b200 import native as N

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", str(rank)))
    if os.environ.get("NCCL_DEBUG", "").upper() in ("WARN", "VERSION"):
        del os.environ["NCCL_DEBUG"]
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    eng = Engine(local_rank)
    if world > 1:
        uid = [eng.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.dist_init(rank, world, uid[0])
    flags = N.RQ_PLAN_PARTITIONED if world > 1 else 0
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
    plan_d = load_plan("micro_join_avg")
    plan = Plan(plan_d)
    if a.micro_cases:
        cases = [(int(float(x.split(":")[0])), int(float(x.split(":")[1]))) for x in a.micro_cases.split(",")]
    else:
        cases = [(10**8, 4), (10**8, 10**6), (10**8, 10**8)]
        if world >= 4:
            cases += [(10**9, 4), (10**9, 10**6), (10**9, 10**8)]
    P_MUL, Q_MUL, Q_ADD = 2654435761, 1000003, 12345           # odd, not multiples of 5: coprime to N = 10^k
    rc = 0
    for n, g in cases:
        if n % 2 == 0 and n % 5 == 0:
            pass
        lo, hi = n * rank // world, n * (rank + 1) // world
        idx = torch.arange(lo, hi, device=dev, dtype=torch.int64)
        foo_a = (idx * P_MUL) % n + 1
        foo_c = ((idx * 2654435769) & 0xFFFFFFFF) % g
        bar_d = (idx * Q_MUL + Q_ADD) % n + 1
        del idx
        cols = {"foo": {"a": foo_a, "c": foo_c}, "bar": {"d": bar_d}}
        tabs = {t["name"]: eng.upload_device(t["name"], {k: (cols[t["name"]][k].data_ptr(), 3, 8) for k in t["columns"]},
                                             hi - lo, borrow=True) for t in plan_d["tables"]}

        def barrier():
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        times, res, tm = [], None, None
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 1 + max(a.warmup, 2) + a.steps
        for i in range(reps):
            barrier()
            t0 = time.perf_counter()
            ev0.record(stream)
            res, tm = eng.execute(plan, tabs, flags)
            ev1.record(stream)
            barrier()
            t = torch.tensor([ev0.elapsed_time(ev1), 1e3 * (time.perf_counter() - t0)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            times.append(t.tolist())
        timed = times[1 + max(a.warmup, 2):]
        if a.dump_outputs and rank == 0:
            dump_outputs(a.dump_outputs, {f"micro_n{n}_g{g}": res}, (64 << 20) // len(cases))
        # ---- independent evaluation ------------------------------------------------------------
        s = torch.zeros(g, dtype=torch.int64, device=dev).index_add_(0, foo_c, foo_a * foo_a)
        k = torch.zeros(g, dtype=torch.int64, device=dev).index_add_(0, foo_c, torch.ones_like(foo_a))
        if world > 1:
            dist.all_reduce(s)
            dist.all_reduce(k)
        keep = k > 0
        want_c = torch.nonzero(keep).flatten()
        num = s[keep] * 100
        want_avg = torch.div(num, k[keep], rounding_mode="trunc")
        got_c = torch.from_numpy(res.columns[0]).to(dev)
        got_avg = torch.from_numpy(res.columns[1]).to(dev)
        ok = res.n_rows == want_c.numel() and bool((got_c == want_c).all()) and bool((got_avg == want_avg).all())
        okt = torch.tensor([int(ok)], device=dev)
        if world > 1:
            dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        ok_all = bool(okt.item())
        if not ok_all:
            rc = 1
        if rank == 0:
            ms = statistics.median([x[0] for x in timed])
            print(json.dumps({
                "metric": "micro_join_groupby_probe_tuples_per_s", "value": n / (ms / 1e3), "unit": "tuples/s", "n_gpus": world,
                "steps": len(timed), "warmup": max(a.warmup, 2), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                "dtype": "int64", "data": "synthetic",
                "config": {"workload": f"README microbenchmark: foo {n} rows join bar {n} rows on a = d, group by c ({g} values), avg(d*a), order by c",
                           "tables": "both row-range sharded, RQ_PLAN_PARTITIONED (hash-partitioned all-to-all)" if world > 1 else "one GPU",
                           "timing": "CUDA events on the engine stream around rq_plan_execute, max over ranks, median of the timed runs"},
                "result_rows": res.n_rows, "checks": {"identical_to_torch_int64_all_ranks": ok_all},
                "first_execution_wall_ms": times[0][1], "wall_ms": statistics.median([x[1] for x in timed]),
                "kernel_ms": tm.kernel_ms, "nccl_ms": tm.nccl_ms, "host_syncs": tm.host_syncs, "gpu_launches": tm.kernel_launches}), flush=True)
        for t in tabs.values():
            t.free()
        del foo_a, foo_c, bar_d, s, k, keep, want_c, num, want_avg, got_c, got_avg, res
        torch.cuda.empty_cache()
    eng.shutdown()
    if world > 1:
        dist.destroy_process_group()
    return rc


# ---------------------------------------------------------------------------------------------
# --workload joins: BASELINE config 3 - the join queries of tpch/queries (Q3, Q5, Q10: HashJoin build /
# probe + GROUP BY + ORDER BY, replicated build sides) at SF10 on one B200. Tables come from the numpy
# generator (all columns the plans touch, strings included), are uploaded through the C ABI, and every
# result is compared with the plan oracle (oracle/plan_oracle.py, pinned to the reference engine) on the
# same data - the checker, not the thing measured. One JSON line per query.
# ---------------------------------------------------------------------------------------------
def main_joins(a):
    import torch
    from resql_b200 import Engine, Plan, tpch
    from oracle.plan_oracle import run_plan
    from common import plan_tables, serialize_columns
    sf = a.sf if a.sf != 100 else 10.0
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    eng = Engine(0)
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
    data = tpch.generate(sf, seed=42, tables=("lineitem", "orders", "customer", "supplier", "nation", "region"))
    n_li = len(data["lineitem"]["l_orderkey"])
    rc = 0
    for q in ("q3", "q5", "q10"):
        d = load_plan(q)
        tabs = plan_tables(d, data)
        t0 = time.perf_counter()
        handles = {n: eng.upload(n, c) for n, c in tabs.items()}
        load_ms = 1e3 * (time.perf_counter() - t0)
        plan = Plan(d)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times, walls = [], []
        reps = 1 + max(a.warmup, 3) + a.steps
        for i in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ev0.record(stream)
            res, tm = eng.execute(plan, handles)
            ev1.record(stream)
            torch.cuda.synchronize()
            times.append(ev0.elapsed_time(ev1)); walls.append(1e3 * (time.perf_counter() - t0))
        timed = times[1 + max(a.warmup, 3):]
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, {q: res}, (64 << 20) // 3)
        got = serialize_columns(res.columns, res.sql_types, res.sql_widths)
        want = serialize_columns(*run_plan(d, tabs))
        order = d.get("order", [])
        keys = lambda lines: [[l.split("|")[c] for c, _ in order[:1]] for l in lines]      # noqa: E731
        # ORDER BY ... LIMIT behind an unstable sort: ties at the cut may differ (qlib/sort.h:21); key sequence + size otherwise
        same = (keys(got) == keys(want) and len(got) == len(want)) if d.get("limit", -1) >= 0 else sorted(got) == sorted(want)
        if not same:
            rc = 1
        ms = statistics.median(timed)
        print(json.dumps({
            "metric": "tpch_join_query_lineitem_tuples_per_s", "value": n_li / (ms / 1e3), "unit": "tuples/s", "n_gpus": 1,
            "steps": len(timed), "warmup": max(a.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "dtype": "int64", "data": "synthetic",
            "config": {"workload": f"TPC-H SF{sf:g} {q} (tpch/queries/{q}.sql), lineitem {n_li} rows, numpy generator seed 42, tables resident",
                       "timing": "CUDA events on the engine stream around rq_plan_execute, median of the timed runs"},
            "result_rows": res.n_rows, "checks": {"identical_to_plan_oracle": bool(same)},
            "first_execution_wall_ms": walls[0], "wall_ms": statistics.median(walls[1 + max(a.warmup, 3):]), "kernel_ms": tm.kernel_ms,
            "host_syncs": tm.host_syncs, "gpu_launches": tm.kernel_launches, "load_ms": load_ms}), flush=True)
        for h in handles.values():
            h.free()
    eng.shutdown()
    return rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (every timed loop runs exactly this many)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sf", type=float, default=float(os.environ.get("RESQL_BENCH_SF", "100")))
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--sample-sf", type=float, default=10.0,
                    help="scale factor of the CPU sample (SF10: 60 M lineitem rows, 8.8 GB in the reference's row format, loaded "
                         "through its binary loader; falls back to SF1 if the box cannot hold it)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--workload", default="tpch", choices=["tpch", "micro", "joins"])
    ap.add_argument("--micro-cases", default="", help="N:G,N:G,... (default: 1e8 x {4,1e6,1e8}; with >= 4 GPUs also 1e9)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the results of the last step as DIR/<query>.<column>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.workload == "micro":
        return main_micro(a)
    if a.workload == "joins":
        return main_joins(a)
    if a.warmup < 3:
        a.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", str(rank)))
    cores = os.cpu_count() or 1

    # ---------------- reference arm: CPU only, rank 0 only ------------------------------------
    if a.impl == "reference":
        if rank != 0:
            return 0
        res = run_reference_with_fallback(a, a.steps + a.warmup, cores)
        if res is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/resql-oracle not built"}))
            return 0
        step_ms = [sum(res["per_query_ms"][q][i] for q in QUERIES) for i in range(a.warmup, a.warmup + a.steps)]
        t = sum(step_ms) / 1e3
        value = 3.0 * res["rows"] * a.steps / t
        sample = f"TPC-H-shaped SF{a.sample_sf} ({res['rows']} lineitem rows), Q1+Q6+Q3, reference JIT, threads={cores}"
        print(json.dumps({
            "impl": "reference", "metric": "tpch_q1_q6_q3_lineitem_tuples_per_s", "value": value, "unit": "tuples/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * t / a.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": f"TPC-H SF{a.sf:g} Q1+Q6+Q3 (bounded CPU sample: SF{a.sample_sf})", "sample": sample},
            "cpu_baseline": {"value": value, "unit": "tuples/s", "cores": cores, "kind": res["kind"], "sample": sample},
            "e2e": {"value": value, "unit": "tuples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "queries": {q: {"ms": statistics.median(res["per_query_ms"][q][a.warmup:]),
                            "tuples_per_s": res["rows"] / (statistics.median(res["per_query_ms"][q][a.warmup:]) / 1e3)} for q in QUERIES},
        }))
        return 0

    # ---------------- our arm --------------------------------------------------------------------
    import torch
    import torch.distributed as dist
    from resql_b200 import Engine, Plan
    from resql_b200 import native as N
    from resql_b200 import tpch_device as TD

    # keep stdout to the one JSON line: NCCL prints its version banner there at WARN/VERSION level
    if os.environ.get("NCCL_DEBUG", "").upper() in ("WARN", "VERSION"):
        del os.environ["NCCL_DEBUG"]
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    eng = Engine(local_rank)
    if world > 1:
        uid = [eng.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.dist_init(rank, world, uid[0])
    flags = N.RQ_PLAN_SHARDED if world > 1 else 0
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)     # the stream the kernels run on

    orders, li, cust = TD.gen_orders_lineitem(a.sf, 42, dev, rank=rank, world=world)
    torch.cuda.synchronize()
    n_local = li["l_orderkey"].numel()
    n_total = n_local
    if world > 1:
        t = torch.tensor([n_local], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        n_total = int(t.item())

    plans = {q: load_plan(q) for q in QUERIES}
    src = {"lineitem": li, "orders": orders, "customer": cust}

    # Resident tables: ONE table per relation, owned by the engine (tile-major pages, see DESIGN.md
    # section 2), holding every column the three plans touch; the plans address columns by name.
    resident = {}
    for name in ("lineitem", "orders", "customer"):
        cols = list(src[name].keys())
        n = src[name][cols[0]].shape[0]
        resident[name] = eng.upload_device(name, TD.as_device_columns(src[name], cols), n, borrow=False)
    torch.cuda.synchronize()
    cplans = {q: Plan(plans[q]) for q in QUERIES}

    # cold start: the very first execution of each plan in this process (empty capacity memos, no
    # recorded host reads, memory pool not grown yet), wall clock around the call - next to the
    # reference's compile time (0.3-1.9 ms asmjit, BASELINE.md) this is our plan-to-result latency
    cold_ms = {}
    for q in QUERIES:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, tm0 = eng.execute(cplans[q], resident, flags)
        cold_ms[q] = {"first_execution_wall_ms": 1e3 * (time.perf_counter() - t0), "lower_ms": tm0.lower_ms,
                      "host_syncs": tm0.host_syncs}

    def step_resident():
        return {q: eng.execute(cplans[q], resident, flags) for q in QUERIES}

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(a.warmup):
        step_resident()
    launches = 0
    per_q = {q: {"kernel_ms": [], "fact_ms": [], "nccl_ms": [], "lower_ms": [], "d2h_ms": [], "host_syncs": []} for q in QUERIES}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        barrier()
        ev0.record(stream)
        for _ in range(a.steps):
            r = step_resident()
            for q in QUERIES:
                tm = r[q][1]
                launches += tm.kernel_launches
                per_q[q]["kernel_ms"].append(tm.kernel_ms)
                per_q[q]["fact_ms"].append(tm.fact_scan_ms)
                per_q[q]["nccl_ms"].append(tm.nccl_ms)
                per_q[q]["lower_ms"].append(tm.lower_ms)
                per_q[q]["d2h_ms"].append(tm.d2h_ms)
                per_q[q]["host_syncs"].append(tm.host_syncs)
        ev1.record(stream)
        barrier()
    dt = max_over_ranks(ev0.elapsed_time(ev1) / 1e3)      # device time on the engine stream
    last = r
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {q: last[q][0] for q in QUERIES})
    clocks = clk.summary()
    value = 3.0 * n_total * a.steps / dt

    # ---- independent check at full size: the same queries evaluated with torch int64 ops -------
    # At N > 1 every rank evaluates its own row range and the partial values are all-reduced
    # (mod-2^64 sums, aggregation.h:182-204: AVG only after the global merge), then compared with
    # the merged result every rank got back from the library. A false check fails the run.
    def allsum(x):
        t = torch.tensor([x], device=dev, dtype=torch.int64) if not torch.is_tensor(x) else x.clone()
        if world > 1:
            dist.all_reduce(t)
        return t

    checks = {}
    m = (li["l_shipdate"] >= 19940101) & (li["l_shipdate"] < 19950101) & (li["l_discount"] >= 5) & \
        (li["l_discount"] <= 7) & (li["l_quantity"] < 24)
    want = int(allsum((li["l_extendedprice"] * li["l_discount"])[m].sum().reshape(1))[0].item())
    got = int(last["q6"][0].columns[0][0]) if last["q6"][0].n_rows else None
    checks["q6_vs_torch"] = (got == want)
    m1 = li["l_shipdate"] <= 19980902
    key = li["l_returnflag"].to(torch.int64) * 256 + li["l_linestatus"].to(torch.int64)
    charge = li["l_extendedprice"] * (100 - li["l_discount"]) * (100 + li["l_tax"])
    res1 = last["q1"][0]
    n_groups_total = int(allsum(torch.unique(key[m1]).numel())[0].item()) if world == 1 else None
    ok = res1.n_rows > 0 and (world > 1 or res1.n_rows == n_groups_total)
    for i in range(res1.n_rows):
        kk = int(res1.columns[0][i]) * 256 + int(res1.columns[1][i])
        sel = m1 & (key == kk)
        part = torch.stack([sel.sum(), charge[sel].sum(), li["l_quantity"][sel].sum(),
                            (li["l_extendedprice"][sel] * (100 - li["l_discount"][sel])).sum(),
                            li["l_discount"][sel].sum()])
        tot = [int(x) for x in allsum(part).tolist()]
        ok &= int(res1.columns[9][i]) == tot[0]
        ok &= int(res1.columns[5][i]) == tot[1]
        ok &= int(res1.columns[2][i]) == tot[2]
        ok &= int(res1.columns[4][i]) == tot[3]
        ok &= tot[0] > 0 and int(res1.columns[8][i]) == (tot[4] * 100) // tot[0]      # AVG after the merge, truncating
    # every valid tuple belongs to exactly one reported group
    ok &= int(sum(int(x) for x in res1.columns[9])) == int(allsum(m1.sum().reshape(1))[0].item())
    checks["q1_vs_torch"] = bool(ok)
    del m, m1, key, charge
    # Q3: top-10 revenue recomputed with torch joins (searchsorted on the unique keys). Orders are
    # range-partitioned with their lineitems (tpch_device), so every order's revenue is complete on
    # one rank: the global top 10 is the top 10 of the ranks' top 10s.
    try:
        cb = cust["c_custkey"][(cust["c_mktsegment"][:, :8] == torch.tensor(list(b"BUILDING"), device=dev, dtype=torch.uint8)).all(1)
                               & (cust["c_mktsegment"][:, 8] == 0)]
        o_ok = (orders["o_orderdate"] < 19950315) & torch.isin(orders["o_custkey"], cb)
        ok_keys, _ = torch.sort(orders["o_orderkey"][o_ok])
        lm = li["l_shipdate"] > 19950315
        lk = li["l_orderkey"][lm]
        pos = torch.searchsorted(ok_keys, lk).clamp(max=max(ok_keys.numel() - 1, 0))
        hit = ok_keys[pos] == lk if ok_keys.numel() else torch.zeros_like(lk, dtype=torch.bool)
        rev = (li["l_extendedprice"][lm] * (100 - li["l_discount"][lm]))[hit]
        uk, inv = torch.unique(lk[hit], return_inverse=True)
        tot = torch.zeros(uk.numel(), dtype=torch.int64, device=dev).index_add_(0, inv, rev)
        top = torch.sort(tot, descending=True).values[:10]
        top = torch.cat([top, torch.full((10 - top.numel(),), -1, dtype=torch.int64, device=dev)])
        if world > 1:
            alltop = [torch.empty_like(top) for _ in range(world)]
            dist.all_gather(alltop, top)
            top = torch.sort(torch.cat(alltop), descending=True).values[:10]
        top = [int(x) for x in top.tolist() if x >= 0]
        res3 = last["q3"][0]
        checks["q3_top10_revenue_vs_torch"] = [int(x) for x in res3.columns[1]] == top
        del o_ok, ok_keys, lm, lk, pos, hit, rev, uk, inv, tot
    except Exception as e:       # the check is independent evidence, never part of the timed path
        checks["q3_top10_revenue_vs_torch"] = f"not run: {e}"
    # all ranks must agree (every rank holds the merged result)
    if world > 1:
        flag = torch.tensor([int(all(v is True for v in checks.values()))], device=dev, dtype=torch.int64)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        checks["all_ranks_agree"] = bool(flag.item() == 1)
    torch.cuda.empty_cache()

    # ---- e2e: host buffers through the C ABI, H2D inside the timed region -------------------------
    e2e = None
    if not a.no_e2e:
        host = {}
        for name in ("lineitem", "orders", "customer"):
            used = []
            for q in QUERIES:
                for t in plans[q]["tables"]:
                    if t["name"] == name:
                        used += [c for c in t["columns"] if c not in used]
            host[name] = {}
            for c in used:
                x = src[name][c]
                hp = torch.empty(x.shape, dtype=x.dtype, pin_memory=True)
                hp.copy_(x)
                host[name][c] = hp
        torch.cuda.synchronize()

        def host_table(name, cols):
            d = {}
            for c in cols:
                arr = host[name][c].numpy()
                if arr.ndim == 2:
                    arr = arr.view(f"S{arr.shape[1]}").reshape(-1)
                d[c] = arr
            return eng.upload(name, d)

        # every step uploads each table ONCE (the union of the columns the three plans scan), runs
        # the three queries on it and reads the results back
        union = {name: list(host[name].keys()) for name in host}

        def host_arrays(name, cols):
            d = {}
            for c in cols:
                arr = host[name][c].numpy()
                if arr.ndim == 2:
                    arr = arr.view(f"S{arr.shape[1]}").reshape(-1)
                d[c] = arr
            return d

        phases = {}

        def step_e2e():
            d2h = 0
            # N > 1: the replicated build sides cross PCIe once (rank 0) and reach the other GPUs over
            # NVLink (rq_table_broadcast); every rank uploads its own lineitem shard
            up = {}
            for name in union:
                t0 = time.perf_counter()
                up[name] = (host_table(name, union[name]) if world == 1 or name == "lineitem"
                            else eng.upload_replicated(name, host_arrays(name, union[name]), 0, rank))
                phases["upload_" + name] = 1e3 * (time.perf_counter() - t0)
            for q in QUERIES:
                t0 = time.perf_counter()
                res, _ = eng.execute(cplans[q], up, flags)
                d2h += sum(c.nbytes for c in res.columns)
                phases["execute_" + q] = 1e3 * (time.perf_counter() - t0)
            t0 = time.perf_counter()
            for h in up.values():
                h.free()
            phases["free"] = 1e3 * (time.perf_counter() - t0)
            return d2h

        for _ in range(2):
            step_e2e()
        e_steps = a.steps
        barrier()
        ev0.record(stream)
        for _ in range(e_steps):
            d2h = step_e2e()
        ev1.record(stream)
        barrier()
        et = max_over_ranks(ev0.elapsed_time(ev1) / 1e3)
        h2d_step = sum(hp.numel() * hp.element_size() for name in host for hp in host[name].values()
                       if world == 1 or name == "lineitem" or rank == 0)
        if world > 1:          # bytes all ranks read from their hosts per step
            tb = torch.tensor([h2d_step], device=dev, dtype=torch.int64)
            dist.all_reduce(tb)
            h2d_step = int(tb.item())
        e2e = {"value": 3.0 * n_total * e_steps / et, "unit": "tuples/s", "h2d_bytes_per_step": int(h2d_step),
               "d2h_bytes_per_step": int(d2h), "steps": e_steps, "ms_per_step": 1e3 * et / e_steps,
               "phases_ms_last_step_rank0": {k: round(v, 2) for k, v in phases.items()},
               "path": "pinned host columns -> rq_table_upload (8-byte columns narrowed on the host cores, H2D, widened on arrival; "
                       "N > 1: replicated tables uploaded by rank 0 and broadcast over NVLink) -> rq_plan_execute -> host result, per step",
               "h2d_bytes_note": "bytes of the host columns in the reference's widths, all ranks; fewer cross PCIe (narrowing)"}
        del host

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 1 if any(v is False for v in checks.values()) else 0

    peak, peak_src = measured_peak()
    traffic_tab = {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic_tab = json.load(f)
    qinfo = {}
    for q in QUERIES:
        fact = statistics.median(per_q[q]["fact_ms"])
        kern = statistics.median(per_q[q]["kernel_ms"])
        gbs = (n_local * BYTES_PER_TUPLE[q]) / (fact / 1e3) / 1e9 if fact > 0 else 0.0
        qinfo[q] = {"kernel_ms": kern, "lineitem_scan_kernel_ms": fact,
                    "nccl_ms": statistics.median(per_q[q]["nccl_ms"]),
                    "lower_ms": statistics.median(per_q[q]["lower_ms"]),
                    "d2h_ms": statistics.median(per_q[q]["d2h_ms"]),
                    "host_syncs_per_execution": statistics.median(per_q[q]["host_syncs"]),
                    "cold": cold_ms[q],
                    "tuples_per_s": n_total / (kern / 1e3) if kern > 0 else None,
                    "algorithmic_bytes_per_tuple": BYTES_PER_TUPLE[q],
                    "lineitem_scan_gbs": gbs, "hbm_frac_of_measured": gbs / peak}
        # whole query: algorithmic bytes of ALL tables the query scans (SURVEY 8d) over ALL its kernels
        wq_bytes = n_total * BYTES_PER_TUPLE[q]
        if q == "q3":
            wq_bytes += 16 * int(src["orders"]["o_orderkey"].shape[0]) + 15 * int(src["customer"]["c_custkey"].shape[0])
        qinfo[q]["whole_query_algorithmic_bytes"] = wq_bytes
        qinfo[q]["whole_query_gbs"] = wq_bytes / world / (kern / 1e3) / 1e9 if kern > 0 else None
        qinfo[q]["whole_query_hbm_frac_of_measured"] = (qinfo[q]["whole_query_gbs"] / peak) if kern > 0 else None
    # dominant kernel = the lineitem scan kernel with the largest share of the step
    dom = max(QUERIES, key=lambda q: qinfo[q]["lineitem_scan_kernel_ms"])
    dom_ms = qinfo[dom]["lineitem_scan_kernel_ms"]
    achieved = qinfo[dom]["lineitem_scan_gbs"]
    traffic = None
    if dom in traffic_tab:
        traffic = traffic_tab[dom]["dram_bytes_per_tuple"] * n_local
    kernel_of = {"q1": "rq_scan_kernel<4> (scan->filter->group->aggregate in registers)",
                 "q6": "rq_scan_kernel<1> (scan->filter->aggregate in registers)",
                 "q3": "rq_scan_kernel<0> (scan->filter->Bloom semi-join->materialize: streaming pass of the two-pass probe)"}
    out = {
        "metric": "tpch_q1_q6_q3_lineitem_tuples_per_s", "value": value, "unit": "tuples/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": f"TPC-H SF{a.sf:g} Q1+Q6+Q3, lineitem {n_total} rows (row-range sharded over {world} GPU), "
                               "dbgen-shaped synthetic generated in HBM, seed 42",
                   "step": "one pass of Q1, Q6 and Q3 over the resident tables (3 lineitem scans + Q3's build and dense probe pipelines)",
                   "l2": "no flush: every query streams >= 14 GB at SF100 (inputs far larger than the 126 MB L2)",
                   "timing": "CUDA events on the engine stream around the K steps, max over ranks"},
        "clocks": clocks, "gpu_launches": launches,
        "roofline": {"bound": "hbm", "kernel": kernel_of[dom], "query": dom,
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "peak_source": peak_src, "algorithmic_bytes_per_tuple": BYTES_PER_TUPLE[dom],
                     "tuples_per_launch": n_local, "launch_ms": dom_ms,
                     "traffic_source": traffic_tab.get(dom, {}).get("source")},
        "queries": qinfo, "checks": checks,
        "step_hbm_frac_of_measured": sum(qinfo[q]["whole_query_algorithmic_bytes"] for q in QUERIES) / world / (dt / a.steps) / 1e9 / peak,
    }
    if e2e is not None:
        out["e2e"] = e2e
    if not a.no_cpu and world == 1:          # (the CPU baseline is reported at N = 1 only)
        try:
            ref = run_reference_with_fallback(a, 3, cores)
            if ref is not None:
                t = sum(statistics.median(ref["per_query_ms"][q]) for q in QUERIES) / 1e3
                out["cpu_baseline"] = {
                    "value": 3.0 * ref["rows"] / t, "unit": "tuples/s", "cores": cores, "kind": ref["kind"],
                    "sample": f"TPC-H-shaped SF{a.sample_sf} ({ref['rows']} lineitem rows), Q1+Q6+Q3, reference JIT threads={cores}, median of 3",
                    "per_query_ms": {q: statistics.median(ref["per_query_ms"][q]) for q in QUERIES}}
        except Exception as e:  # the baseline is reported, never required for the GPU number
            out["cpu_baseline"] = {"value": None, "unit": "tuples/s", "cores": cores, "kind": "reference", "sample": f"failed: {e}"}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    bad = [k for k, v in checks.items() if v is False]
    if bad:
        print(f"bench.py: result check(s) failed: {bad}", file=sys.stderr)
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
