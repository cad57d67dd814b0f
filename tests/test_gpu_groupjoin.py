"""Groupjoin (engine_exec.inl groupjoin_probe): a GROUP BY on the key of a direct-address join
aggregates into the join's entries. Q3 and Q3-shaped plans must give the oracle's result with the
groupjoin on and off, and the groupjoin must run exactly where it is eligible (fewer launches: no
hash-table init)."""
import copy

import numpy as np
import pytest

from common import load_plan_dict, plan_tables, serialize_columns, assert_same_relation
from oracle.plan_oracle import run_plan
from resql_b200 import Plan, tpch

pytestmark = pytest.mark.gpu

INT, BIGINT, DECIMAL, DATE = 3, 4, 5, 7
SUM, COUNT, MIN, MAX = 1, 2, 3, 4


@pytest.fixture(scope="module")
def engine():
    from resql_b200 import Engine
    eng = Engine(0)
    yield eng
    eng.shutdown()


@pytest.fixture(scope="module")
def data():
    return tpch.generate(0.06, seed=2026, tables=("lineitem", "orders", "customer"))


def _run(engine, d, tabs, group_joins):
    """careful execution (no replay: the option must take effect) -> (rows, kernel launches)"""
    engine.set_option("group_joins", group_joins)
    engine.set_option("replay", 0)
    handles = {n: engine.upload(n, c) for n, c in tabs.items()}
    try:
        res, tm = engine.execute(Plan(d), handles)
    finally:
        for h in handles.values():
            h.free()
        engine.set_option("group_joins", 1)
        engine.set_option("replay", 1)
    return serialize_columns(res.columns, res.sql_types, res.sql_widths), tm.kernel_launches


def _check(engine, d, tabs, what, eligible):
    """both paths give the oracle's result; eligible True / False: the groupjoin runs / does not run
    (launch counts of the second execution of each path, once the pipeline memos know the tables)"""
    want = serialize_columns(*run_plan(d, tabs))
    launches = {}
    for group_joins in (1, 0, 1, 0):
        got, launches[group_joins] = _run(engine, d, tabs, group_joins)
        assert_same_relation(got, want, d, what + (" (groupjoin)" if group_joins else " (hash aggregation)"))
    if eligible is True:
        assert launches[1] < launches[0], f"{what}: the groupjoin did not run ({launches[1]} vs {launches[0]} launches)"
    elif eligible is False:
        assert launches[1] == launches[0], f"{what}: launches differ ({launches[1]} vs {launches[0]}) on the same path"


def _q3_variant(keys=None, vals=None, extra_nodes=()):
    """Q3 with other GROUP BY keys / aggregates in its lineitem pipeline, followed by a projection of all
    of its columns (no ORDER BY). Lineitem nodes: 0 l_orderkey, 1 l_extendedprice, 2 l_discount,
    7 PROBE orders, 8 PAYLOAD o_orderkey, 9 o_orderdate, 10 o_shippriority, 15 revenue."""
    d = copy.deepcopy(load_plan_dict("q3"))
    p = d["pipelines"][2]
    p["nodes"] += [list(n) for n in extra_nodes]
    if keys is not None:
        p["keys"] = [list(k) for k in keys]
    if vals is not None:
        p["vals"] = [list(v) for v in vals]
    cols = p["keys"] + p["vals"]
    d["pipelines"][3] = {"source_kind": 2, "source_id": 2, "source_id2": 0, "sink_kind": 3, "size_hint": 0,
                         "nodes": [[1, c, 0, 0, 0] for c in range(len(cols))], "args": [], "keys": [],
                         "vals": [[c, 0, v[2], v[3]] for c, v in enumerate(cols)]}
    d["order"] = []
    d["limit"] = -1
    d["result_names"] = [f"c{c}" for c in range(len(cols))]
    d["result_types"] = ["BIGINT"] * len(cols)
    return d


Q3_KEYS = [[0, 0, INT, 0], [9, 0, DATE, 0], [10, 0, INT, 0]]


@pytest.mark.parametrize("rows", [0, 1, 1023, 1025, 300_001])
def test_q3_sizes(rows, engine, data):
    d = load_plan_dict("q3")
    tabs = plan_tables(d, data)
    tabs["lineitem"] = {c: v[:rows] for c, v in tabs["lineitem"].items()}
    _check(engine, d, tabs, f"q3@{rows}", eligible=True if rows > 0 else None)


def test_q3_empty_join(engine, data):
    """no lineitem key has an order: every probe misses, the result is empty"""
    d = load_plan_dict("q3")
    tabs = plan_tables(d, data)
    tabs["lineitem"] = dict(tabs["lineitem"])
    tabs["lineitem"]["l_orderkey"] = (tabs["lineitem"]["l_orderkey"] + 1_000_000_000).astype(tabs["lineitem"]["l_orderkey"].dtype)
    _check(engine, d, tabs, "q3 empty join", eligible=None)     # (the pruned build may be empty)


def test_count_min_max_with_negative_values(engine, data):
    # 16 = l_discount - l_extendedprice (negative), 18 = l_orderkey - 3 000 000 (both signs)
    d = _q3_variant(keys=Q3_KEYS,
                    vals=[[15, SUM, DECIMAL, 4868], [0, COUNT, BIGINT, 0], [16, MIN, DECIMAL, 3074], [16, MAX, DECIMAL, 3074],
                          [18, MIN, BIGINT, 0], [18, MAX, BIGINT, 0], [15, SUM, DECIMAL, 4868]],
                    extra_nodes=[[5, 2, 1, 0, 0], [2, 0, 0, 0, 3_000_000], [5, 0, 17, 0, 0]])
    _check(engine, d, plan_tables(d, data), "q3 count/min/max", eligible=True)


def test_avg(engine, data):
    """AVG is SUM and COUNT in the aggregation, divided by the projection behind it"""
    d = _q3_variant(keys=Q3_KEYS, vals=[[15, SUM, DECIMAL, 4868], [0, COUNT, BIGINT, 0]])
    d["pipelines"][3]["nodes"] = [[1, 0, 0, 0, 0], [1, 3, 0, 0, 0], [1, 4, 0, 0, 0], [2, 0, 0, 0, 100],
                                  [6, 1, 3, 0, 0], [7, 4, 2, 0, 0]]
    d["pipelines"][3]["vals"] = [[0, 0, INT, 0], [5, 0, DECIMAL, 4868]]
    d["result_names"] = ["l_orderkey", "avg_revenue"]
    d["result_types"] = ["INT", "DECIMAL(19,4)"]
    _check(engine, d, plan_tables(d, data), "q3 avg", eligible=True)


def test_join_key_repeat_as_key(engine, data):
    d = _q3_variant(keys=[[8, 0, INT, 0], [9, 0, DATE, 0], [10, 0, INT, 0]])
    _check(engine, d, plan_tables(d, data), "q3 keyed by o_orderkey", eligible=True)


def test_probe_keys_outside_the_build_domain(engine, data):
    d = load_plan_dict("q3")
    tabs = plan_tables(d, data)
    li = dict(tabs["lineitem"])
    k = li["l_orderkey"].astype(np.int64).copy()
    k[::7] += 10_000_000
    k[3::11] = -k[3::11]
    li["l_orderkey"] = k.astype(li["l_orderkey"].dtype)
    tabs["lineitem"] = li
    _check(engine, d, tabs, "q3 probe keys outside the domain", eligible=True)


def test_unsorted_probe_keys(engine, data):
    d = load_plan_dict("q3")
    tabs = plan_tables(d, data)
    perm = np.random.default_rng(5).permutation(len(tabs["lineitem"]["l_orderkey"]))
    tabs["lineitem"] = {c: np.ascontiguousarray(v[perm]) for c, v in tabs["lineitem"].items()}
    _check(engine, d, tabs, "q3 unsorted lineitem", eligible=True)


def test_duplicate_build_keys_take_the_hash_path(engine, data):
    """a duplicate o_orderkey makes the build take the hash form: no groupjoin, same result"""
    d = load_plan_dict("q3")
    tabs = plan_tables(d, data)
    o = tabs["orders"]
    dup = np.arange(0, len(o["o_orderkey"]), 97)
    tabs["orders"] = {c: np.concatenate([v, v[dup]]) for c, v in o.items()}
    _check(engine, d, tabs, "q3 duplicate orders", eligible=False)


def test_key_set_without_the_join_key(engine, data):
    d = _q3_variant(keys=[[9, 0, DATE, 0], [10, 0, INT, 0]])
    _check(engine, d, plan_tables(d, data), "q3 grouped by orderdate, shippriority", eligible=False)


def test_replayed_and_graph_executions(engine, data):
    d = load_plan_dict("q3")
    tabs = plan_tables(d, data)
    want = serialize_columns(*run_plan(d, tabs))
    handles = {n: engine.upload(n, c) for n, c in tabs.items()}
    try:
        runs = []
        p = Plan(d)
        for _ in range(6):           # careful, careful, replay, replay + capture, graph, graph
            res, tm = engine.execute(p, handles)
            runs.append((serialize_columns(res.columns, res.sql_types, res.sql_widths), tm))
    finally:
        for h in handles.values():
            h.free()
    for got, _ in runs:
        assert_same_relation(got, want, d, "q3 (repeated)")
    assert runs[-1][1].host_syncs == 1, f"replay waited {runs[-1][1].host_syncs} times"
