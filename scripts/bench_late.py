#!/usr/bin/env python
"""Late materialization benchmark: `select * from lineitem, orders where l_orderkey = o_orderkey and
l_shipdate < D` (25 columns, the late form) with D keeping 100 %, 10 %, 1 % and 0.01 % of lineitem,
and a 24-column shape both forms run (the same join without o_comment), early against forced late
(`late_materialize` 2).

    python scripts/bench_late.py [--sf 10] [--reps 5]

Per case one JSON line: median and minimum over --reps timed executions (after one warm-up) of the
kernel time the engine reports (rq_timings.kernel_ms: the scan, the gather and the result kernels),
of the fact-table scan kernel alone (scan_kernel_ms) and of the execute call; output rows/s from the
median kernel time; the bytes of the output columns (8 per value, what the scan and the gather write);
and the card's name and power limit. Every result is checked against an independent numpy evaluation:
the row count, and sums of l_orderkey, l_extendedprice, o_totalprice and o_custkey over the result."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
    name, plim = [x.strip() for x in out.split(",")]
    return name, plim


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sf", type=float, default=10)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    from resql_b200 import Engine, Plan, tpch
    from test_gpu_late_materialize import LT, lineitem_orders, schema, tp_tabs
    card, plim = gpu_info()
    data = tpch.generate(a.sf, seed=1, tables=("lineitem", "orders"))
    tabs = tp_tabs(data, ("orders", "lineitem"))
    eng = Engine(0)
    handles = {n: eng.upload(n, c) for n, c in tabs.items()}
    L, O = data["lineitem"], data["orders"]
    sd = np.sort(L["l_shipdate"])
    opos = np.searchsorted(O["o_orderkey"], L["l_orderkey"])        # orders are generated in key order
    assert (O["o_orderkey"][opos] == L["l_orderkey"]).all()

    def expect(mask):
        s = lambda x: int(x[mask].astype(np.int64).sum(dtype=np.int64))
        return [int(mask.sum()), s(L["l_orderkey"]), s(L["l_extendedprice"]), s(O["o_totalprice"][opos]), s(O["o_custkey"][opos])]

    def run(d, mode, label, frac, cutoff):
        eng.set_option("late_materialize", mode)
        p = Plan(d)
        res, _ = eng.execute(p, handles)
        ks, ss, ws = [], [], []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            res, tm = eng.execute(p, handles)
            ws.append((time.perf_counter() - t0) * 1e3)
            ks.append(tm.kernel_ms); ss.append(tm.scan_kernel_ms)
        ncols = len(res.columns)
        got = [res.n_rows if hasattr(res, "n_rows") else len(res.columns[0])]
        got += [int(res.columns[c].astype(np.int64).sum(dtype=np.int64)) for c in (0, 5, 16 + 3, 16 + 1)]
        want = expect(L["l_shipdate"] < cutoff)
        k = statistics.median(ks)
        print(json.dumps({"case": label, "form": ["early", "default", "late"][mode], "frac": frac, "columns": ncols,
                          "rows": got[0], "ok": got == want, "kernel_ms": round(k, 3), "kernel_ms_min": round(min(ks), 3),
                          "scan_ms": round(statistics.median(ss), 3), "execute_ms": round(statistics.median(ws), 3),
                          "rows_per_s": got[0] / (k * 1e-3) if k > 0 else None, "bytes_written": got[0] * ncols * 8,
                          "sf": a.sf, "card": card, "power_limit": plim}), flush=True)
        assert got == want, (label, got, want)

    for frac in (1.0, 0.1, 0.01, 0.0001):
        cutoff = int(sd[min(int(frac * len(sd)), len(sd) - 1)]) + (1 if frac == 1.0 else 0)
        run(lineitem_orders([(LT, 10, cutoff)]), 1, "select_star_25", frac, cutoff)
    for frac in (1.0, 0.01):
        cutoff = int(sd[min(int(frac * len(sd)), len(sd) - 1)]) + (1 if frac == 1.0 else 0)
        d = lineitem_orders([(LT, 10, cutoff)])
        d["pipelines"][1]["vals"] = d["pipelines"][1]["vals"][:-1]     # without o_comment: 24 columns
        d["result_names"], d["result_types"] = d["result_names"][:-1], d["result_types"][:-1]
        for mode in (1, 2):
            run(d, mode, "select_24", frac, cutoff)
    for h in handles.values():
        h.free()
    eng.shutdown()


if __name__ == "__main__":
    main()
