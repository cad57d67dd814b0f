#!/usr/bin/env python
"""Nested-loops join benchmark: the `nlj_noneq_group` shape (customer x orders under a non-equi
condition, grouped by market segment) at 2^20 ... 2^36 pairs, plus one selective materialize.

    python scripts/bench_nlj.py [--tree DIR] [--label NAME] [--log2-pairs 20,24,28,32,36] [--reps N]

The children are seeded TPC-H-shaped columns (customer: c_acctbal, c_mktsegment as its code 0-4;
orders: o_totalprice, o_orderdate), materialized by two scan pipelines; the third pipeline is
the NLJ:
    agg:   select c_mktsegment, count(*), min(o_orderdate) where c_acctbal * 20 > o_totalprice
           group by c_mktsegment
    emit:  select c_acctbal, o_orderdate where o_totalprice < c_acctbal * 2     (about 2 % of pairs)
Every result is checked against a numpy evaluation that never builds the product (orders sorted by
o_totalprice, searchsorted, prefix minima / sums). Per case one JSON line: the median and minimum
over --reps timed executions (after one warm-up) of the kernel time the engine reports
(rq_timings.kernel_ms, all kernels of the plan including the two child scans) and of the wall time
of the execute call, pairs/s from the median kernel time, and the card's name and power limit.
--tree runs the library of another checkout (e.g. the parent commit) with the same inputs; a size
that build refuses prints its error instead of a time. Orders has 16x the rows of customer."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

SELF_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M64 = (1 << 64) - 1


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
        name, plim = [x.strip() for x in out.split(",")]
        return name, plim
    except Exception as e:       # (a machine without nvidia-smi still benchmarks; the fields say so)
        return f"unknown ({e})", "unknown"


def children(nl, nr, seed):
    rng = np.random.default_rng(seed)
    cust = {"c_acctbal": rng.integers(-99_999, 1_000_000, nl, dtype=np.int64),           # DECIMAL(12,2) cents
            "c_mktsegment": rng.integers(0, 5, nl, dtype=np.int64)}
    orders = {"o_totalprice": rng.integers(90_000, 50_000_000, nr, dtype=np.int64),
              "o_orderdate": rng.integers(8035, 10_591, nr, dtype=np.int64)}           # 1992-01-01 .. 1998-12-31
    return cust, orders


def plan(case):
    def scan(tid, ncol):
        return {"source_kind": 1, "source_id": tid, "source_id2": 0, "sink_kind": 3, "size_hint": 0,
                "nodes": [[1, c, 0, 0, 0] for c in range(ncol)], "args": [], "keys": [],
                "vals": [[c, 0, 4, 0] for c in range(ncol)]}
    # columns of the cross source: 0 c_acctbal, 1 c_mktsegment, 2 o_totalprice, 3 o_orderdate
    cols = [[1, c, 0, 0, 0] for c in range(4)]
    if case == "agg":
        nlj = {"source_kind": 3, "source_id": 0, "source_id2": 1, "sink_kind": 1, "size_hint": 5,
               "nodes": cols + [[2, 0, 0, 0, 20], [6, 0, 4, 0, 0], [12, 5, 2, 0, 0], [22, 6, 0, 0, 0]],
               "args": [], "keys": [[1, 0, 4, 0]], "vals": [[0, 2, 4, 0], [3, 3, 4, 0]]}
    else:
        nlj = {"source_kind": 3, "source_id": 0, "source_id2": 1, "sink_kind": 3, "size_hint": 0,
               "nodes": cols + [[2, 0, 0, 0, 2], [6, 0, 4, 0, 0], [10, 2, 5, 0, 0], [22, 6, 0, 0, 0]],
               "args": [], "keys": [], "vals": [[0, 0, 4, 0], [3, 0, 4, 0]]}
    return {"tables": [{"name": "customer", "columns": ["c_acctbal", "c_mktsegment"]},
                       {"name": "orders", "columns": ["o_totalprice", "o_orderdate"]}],
            "pipelines": [scan(0, 2), scan(1, 2), nlj], "order": [], "limit": -1, "strpool": "",
            "result_names": ["a", "b", "c"][: 3 if case == "agg" else 2], "result_types": ["BIGINT"] * (3 if case == "agg" else 2)}


def reference(case, cust, orders):
    o = np.argsort(orders["o_totalprice"], kind="stable")
    tp = orders["o_totalprice"][o]
    if case == "agg":
        # orders with o_totalprice < 20 * c_acctbal: a prefix of the sorted orders
        cnt = np.searchsorted(tp, cust["c_acctbal"] * 20, side="left")
        pmin = np.concatenate([[np.iinfo(np.int64).max], np.minimum.accumulate(orders["o_orderdate"][o])])
        res = {}
        for g in range(5):
            m = cust["c_mktsegment"] == g
            c = int(cnt[m].sum())
            if c:
                res[g] = (c, int(pmin[cnt[m]].min()))
        return res
    cnt = np.searchsorted(tp, cust["c_acctbal"] * 2, side="left")
    psum = np.concatenate([[0], np.cumsum(orders["o_orderdate"][o].astype(np.uint64), dtype=np.uint64)])
    n = int(cnt.sum())
    s_acct = int((cust["c_acctbal"].astype(np.uint64) * cnt.astype(np.uint64)).sum(dtype=np.uint64))
    s_date = int(psum[cnt].sum(dtype=np.uint64))
    return n, s_acct & M64, s_date & M64


def observed(case, cols):
    if case == "agg":
        return {int(k): (int(c), int(d)) for k, c, d in zip(*cols)}
    return (len(cols[0]), int(cols[0].astype(np.uint64).sum(dtype=np.uint64)) & M64,
            int(cols[1].astype(np.uint64).sum(dtype=np.uint64)) & M64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=SELF_ROOT, help="checkout whose resql_b200 (and built library) is measured")
    ap.add_argument("--label", default="this")
    ap.add_argument("--log2-pairs", default="20,24,28,32,36")
    ap.add_argument("--emit-log2-pairs", type=int, default=28)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=2026)
    a = ap.parse_args()
    sys.path.insert(0, os.path.abspath(a.tree))
    from resql_b200 import Engine, EngineError, Plan
    name, plim = gpu_info()
    eng = Engine(0)
    cases = [("agg", int(k)) for k in a.log2_pairs.split(",") if k] + [("emit", a.emit_log2_pairs)]
    for case, lg in cases:
        nl = 1 << ((lg - 4) // 2)
        nr = (1 << lg) // nl                     # orders : customer = 16 : 1 for even exponents
        cust, orders = children(nl, nr, a.seed + lg)
        rec = {"build": a.label, "case": case, "log2_pairs": lg, "pairs": nl * nr, "customer_rows": nl,
               "orders_rows": nr, "gpu": name, "power_limit": plim}
        hc, ho = eng.upload("customer", cust), eng.upload("orders", orders)
        try:
            p = Plan(plan(case))
            want = reference(case, cust, orders)
            kms, wall = [], []
            for r in range(a.reps + 1):
                t0 = time.perf_counter()
                res, tm = eng.execute(p, {"customer": hc, "orders": ho})
                w = (time.perf_counter() - t0) * 1e3
                if r == 0:
                    rec["ok"] = observed(case, res.columns) == want
                else:
                    kms.append(tm.kernel_ms)
                    wall.append(w)
                if r == 0 and not rec["ok"]:
                    break
            if kms:
                med = statistics.median(kms)
                rec.update(kernel_ms=round(med, 4), kernel_ms_min=round(min(kms), 4),
                           wall_ms=round(statistics.median(wall), 4), pairs_per_s=nl * nr / (med * 1e-3),
                           result_rows=len(res.columns[0]))
        except EngineError as e:
            rec.update(status="refused", error=str(e))
        finally:
            hc.free()
            ho.free()
        print(json.dumps(rec), flush=True)
    eng.shutdown()


if __name__ == "__main__":
    main()
