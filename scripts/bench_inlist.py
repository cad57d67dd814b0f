#!/usr/bin/env python
"""IN-list benchmark: `select sum(l_extendedprice) from lineitem where <list>` on resident SF10 lineitem,
with l_partkey lists of 2, 4, 8 and 11 values unrolled (`in_lists` 0) and as one set test (`in_lists` 2),
64, 1024 and 10^5 values as a set test (the old form cannot lower them), and l_shipmode CHAR lists of 2
and 7 values in both forms.

    python scripts/bench_inlist.py [--sf 10] [--reps 10]

Per case one JSON line: median and minimum over --reps timed executions (after one warm-up) of the kernel
time the engine reports (rq_timings.kernel_ms), the set form the host chose, and the card's name and
power limit. Every result is checked against numpy."""
import argparse
import json
import os
import statistics
import subprocess
import sys

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
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    from resql_b200 import Engine, Plan, tpch
    import inlist_plans as IP
    card, plim = gpu_info()
    cols = ["l_partkey", "l_extendedprice", "l_shipmode"]
    L = tpch.generate(a.sf, seed=1, tables=("lineitem",))["lineitem"]
    eng = Engine(0)
    h = eng.upload("lineitem", {c: L[c] for c in cols})
    rng = np.random.default_rng(5)
    keys = np.unique(L["l_partkey"])

    def run(label, col, consts, eq, mode):
        eng.set_option("in_lists", mode)
        d = IP.sum_in("lineitem", cols, col, consts, "l_extendedprice", eq=eq)
        p = Plan(d)
        res, _ = eng.execute(p, {"lineitem": h})
        ks = []
        for _ in range(a.reps):
            res, tm = eng.execute(p, {"lineitem": h})
            ks.append(tm.kernel_ms)
        if eq == "EQ":
            m = np.isin(L[col], np.array(consts))
        else:
            cs = set(c.encode() for c in consts)
            m = np.array([v.rstrip(b" ") in cs for v in L[col]])
        want = (int(L["l_extendedprice"][m].astype(np.int64).sum()), int(m.sum()))
        got = (int(res.columns[0][0]), int(res.columns[1][0])) if res.n_rows else (0, 0)
        print(json.dumps({"case": label, "values": len(consts), "form": ["unrolled", "default", "set"][mode],
                          "rows": want[1], "ok": got == want, "kernel_ms": round(statistics.median(ks), 4),
                          "kernel_ms_min": round(min(ks), 4), "sf": a.sf, "card": card, "power_limit": plim}), flush=True)
        assert got == want, (label, got, want)

    for k in (2, 4, 8, 11):
        consts = [int(x) for x in rng.choice(keys, k, replace=False)]
        for mode in (0, 2):
            run("l_partkey", "l_partkey", consts, "EQ", mode)
    for k in (64, 1024, 100000):
        run("l_partkey", "l_partkey", [int(x) for x in rng.choice(keys, k, replace=False)], "EQ", 2)
    for consts in (["MAIL", "SHIP"], ["MAIL", "SHIP", "AIR", "REG AIR", "RAIL", "TRUCK", "FOB"]):
        for mode in (0, 2):
            run("l_shipmode", "l_shipmode", consts, "EQ_CHAR", mode)
    h.free()
    eng.shutdown()


if __name__ == "__main__":
    main()
