"""IN lists on the B200: OR trees of equality tests against constants run as one set-membership unit of the
scan kernel (bitmap, sorted array or string table), in every kernel variant and pipeline shape, against
the plan oracle or numpy. Lists of 12 values and more were refused before (more live values than slots)."""
import numpy as np
import pytest

from common import plan_tables, serialize_columns, assert_same_relation
from oracle.plan_oracle import run_plan
from resql_b200 import Plan
import inlist_plans as IP

pytestmark = pytest.mark.gpu

LI = ["l_orderkey", "l_partkey", "l_linenumber", "l_quantity", "l_extendedprice", "l_discount", "l_returnflag",
      "l_shipdate", "l_shipmode", "l_shipinstruct"]
OR_ = ["o_orderkey", "o_custkey", "o_totalprice", "o_orderdate", "o_orderpriority", "o_clerk"]
PA = ["p_partkey", "p_brand", "p_size", "p_container"]
OUT = [("l_orderkey", IP.SQL_INT, 0), ("l_extendedprice", IP.SQL_BIGINT, 0)]


@pytest.fixture(scope="module")
def engine():
    from resql_b200 import Engine
    eng = Engine(0)
    yield eng
    eng.set_option("in_lists", 1)
    eng.shutdown()


@pytest.fixture(scope="module")
def gpu_tabs(engine, sf001):
    up = {"lineitem": engine.upload("lineitem", {c: sf001["lineitem"][c] for c in LI}),
          "orders": engine.upload("orders", {c: sf001["orders"][c] for c in OR_}),
          "part": engine.upload("part", {c: sf001["part"][c] for c in PA})}
    yield up
    for h in up.values():
        h.free()


@pytest.fixture(autouse=True)
def default_options(engine):
    yield
    for k, v in (("in_lists", 1), ("late_materialize", 1), ("split_min_rows", -1), ("split_frac", -1)):
        engine.set_option(k, v)


def execute(engine, gpu_tabs, d):
    res, tm = engine.execute(Plan(d), {t["name"]: gpu_tabs[t["name"]] for t in d["tables"]})
    return serialize_columns(res.columns, res.sql_types, res.sql_widths), res, tm


def against_oracle(engine, gpu_tabs, sf001, d, what=""):
    want = serialize_columns(*run_plan(d, plan_tables(d, sf001)))
    got, _, _ = execute(engine, gpu_tabs, d)
    assert_same_relation(got, want, d, what)
    return len(want)


def int_consts(col_values, k, seed, extra=()):
    rng = np.random.default_rng(seed)
    u = np.unique(col_values)
    pick = [int(x) for x in rng.choice(u, size=min(k, len(u)), replace=False)]
    while len(pick) < k:
        pick.append(int(rng.integers(-10 ** 6, 10 ** 9)))
    return pick + list(extra)


def agg_vs_numpy(engine, gpu_tabs, sf001, table, cols, tested, consts, summed, group=None):
    d = IP.sum_in(table, cols, tested, consts, summed, group=group)
    got, res, _ = execute(engine, gpu_tabs, d)
    T = sf001[table]
    m = np.isin(np.asarray(T[tested]).astype(np.int64), np.array(consts, dtype=np.int64))
    if group is None:
        s = int(np.asarray(T[summed])[m].astype(np.int64).sum())
        n = int(m.sum())
        if n == 0:
            assert res.n_rows == 0 or int(res.columns[1][0]) == 0
        else:
            assert (int(res.columns[0][0]), int(res.columns[1][0])) == (s, n), (tested, len(consts))
    else:
        g = np.asarray(T[group])[m]
        want = {int(k): (int(np.asarray(T[summed])[m][g == k].astype(np.int64).sum()), int((g == k).sum())) for k in np.unique(g)}
        have = {int(res.columns[0][i]): (int(res.columns[1][i]), int(res.columns[2][i])) for i in range(res.n_rows)}
        assert have == want
    return int(m.sum())


# ---- integer lists ------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 11, 12, 64, 65, 1000, 100000])
@pytest.mark.parametrize("col", ["l_linenumber", "l_partkey", "l_orderkey", "l_returnflag"])
def test_integer_lists_lineitem(engine, gpu_tabs, sf001, col, k):
    consts = int_consts(sf001["lineitem"][col], k, k, extra=(-7, 2 ** 40, -(2 ** 33), 0))
    consts += consts[: k // 3]                                          # duplicates
    agg_vs_numpy(engine, gpu_tabs, sf001, "lineitem", LI, col, consts, "l_extendedprice")


@pytest.mark.parametrize("k", [2, 12, 1000])
def test_integer_lists_totalprice(engine, gpu_tabs, sf001, k):
    consts = int_consts(sf001["orders"]["o_totalprice"], k, 3, extra=(-5,))
    assert agg_vs_numpy(engine, gpu_tabs, sf001, "orders", OR_, "o_totalprice", consts, "o_custkey") > 0


def test_list_without_matches(engine, gpu_tabs, sf001):
    assert agg_vs_numpy(engine, gpu_tabs, sf001, "lineitem", LI, "l_partkey", [-1, -2, 10 ** 9, 10 ** 9 + 1] * 5,
                        "l_extendedprice") == 0
    d = IP.select_in("lineitem", LI, "l_partkey", list(range(-40, -1)), OUT)
    assert against_oracle(engine, gpu_tabs, sf001, d) == 0


# l_partkey spans 2000 values at this scale (every list is a bitmap); l_orderkey 60000 (a sparse list is sorted)
@pytest.mark.parametrize("col,consts", [("l_partkey", list(range(100, 4000, 3))), ("l_orderkey", [i * 797 for i in range(1, 76)])],
                         ids=["bitmap", "sorted"])
@pytest.mark.parametrize("shape", ["right", "left", "balanced"])
def test_set_forms_and_shapes(engine, gpu_tabs, sf001, col, consts, shape):
    d = IP.select_in("lineitem", LI, col, consts, OUT, shape)
    assert against_oracle(engine, gpu_tabs, sf001, d) > 0


def test_computed_value(engine, gpu_tabs, sf001):
    d = IP.select_in("lineitem", LI, "l_linenumber", [2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37], OUT, computed=True)
    assert against_oracle(engine, gpu_tabs, sf001, d) > 0


# ---- string lists -------------------------------------------------------------------------------------
STRS = ["MAIL", "AIR  ", "REG AIR", "", "TRUCK     XX", "TRUCK", "SHIP", "SHIP", "NONE ", "DELIVER IN PERSON",
        "TAKE BACK RETURN AND MORE THAN THE COLUMN HOLDS", "COLLECT COD", "COLLECT CO", "COLLECT CODX"]


@pytest.mark.parametrize("eq", ["EQ_CHAR", "EQ_VARCHAR"])
@pytest.mark.parametrize("col", ["l_shipmode", "l_shipinstruct"])
def test_string_lists(engine, gpu_tabs, sf001, eq, col):
    d = IP.select_in("lineitem", LI, col, STRS, OUT, "right", eq)
    assert against_oracle(engine, gpu_tabs, sf001, d) > 0


@pytest.mark.parametrize("eq", ["EQ_CHAR", "EQ_VARCHAR"])
def test_string_lists_with_blanks_in_data(engine, sf001, eq):
    # trailing blanks in the data: CHAR ignores them, VARCHAR does not; the empty string; long shared prefixes
    vals = np.array([b"AB", b"AB  ", b"", b"   ", b"PREFIX-PREFIX-PREFIX-1", b"PREFIX-PREFIX-PREFIX-2", b"ABC", b"A"] * 300, dtype="S24")
    ids = np.arange(len(vals), dtype=np.int64)
    h = engine.upload("t", {"s": vals, "i": ids})
    try:
        for consts in (["AB", "", "PREFIX-PREFIX-PREFIX-2", "PREFIX-PREFIX-PREFIX-", "X"], ["AB  ", "   ", "A  "]):
            d = IP.select_in("t", ["s", "i"], "s", consts, [("i", IP.SQL_BIGINT, 0)], "right", eq)
            want = serialize_columns(*run_plan(d, {"t": {"s": vals, "i": ids}}))
            res, _ = engine.execute(Plan(d), {"t": h})
            assert_same_relation(serialize_columns(res.columns, res.sql_types, res.sql_widths), want, d, eq)
    finally:
        h.free()


def test_thousand_strings(engine, gpu_tabs, sf001):
    consts = [f"Clerk#{i:09d}" for i in range(1, 2000, 2)]
    d = IP.select_in("orders", OR_, "o_clerk", consts, [("o_orderkey", IP.SQL_INT, 0)], "balanced", "EQ_CHAR")
    got, res, _ = execute(engine, gpu_tabs, d)
    cs = set(c.encode() for c in consts)
    want = np.sort(np.asarray(sf001["orders"]["o_orderkey"])[[c.rstrip(b" ") in cs for c in sf001["orders"]["o_clerk"]]])
    assert len(want) > 0 and np.array_equal(np.sort(np.asarray(res.columns[0]).astype(np.int64)), want)


# ---- placements ---------------------------------------------------------------------------------------
def test_in_case(engine, gpu_tabs, sf001):
    d = IP.case_in("lineitem", LI, "l_partkey", int_consts(sf001["lineitem"]["l_partkey"], 40, 1), "l_extendedprice")
    against_oracle(engine, gpu_tabs, sf001, d)
    d = IP.case_in("lineitem", LI, "l_shipmode", STRS, "l_quantity", eq="EQ_CHAR")
    against_oracle(engine, gpu_tabs, sf001, d)


def test_two_lists_ored(engine, gpu_tabs, sf001):
    d = IP.two_lists("lineitem", LI, "l_linenumber", [1, 7], "l_partkey", int_consts(sf001["lineitem"]["l_partkey"], 30, 4), OUT)
    assert against_oracle(engine, gpu_tabs, sf001, d) > 0


CONTAINERS = [f"{s} {c}" for s in ("SM", "MED", "LG", "JUMBO", "WRAP") for c in ("CASE", "BOX", "BAG", "JAR", "PKG", "PACK", "CAN", "DRUM")]


def q19_shape(n_containers=20):
    """Q19 with 20-value container lists on the probe's string payload, inside AND / OR arms"""
    d, pool = IP.new_plan({"part": PA, "lineitem": LI})
    b = IP.Pipe(d, "part", PA, pool)
    cols = [b.col(c) for c in PA]
    b.done(IP.SINK_BUILD, [[cols[0], 0, IP.SQL_INT, 0], [cols[1], 0, IP.SQL_CHAR, 10], [cols[2], 0, IP.SQL_INT, 0],
                           [cols[3], 0, IP.SQL_CHAR, 10]], keys=[[cols[0], 0, IP.SQL_INT, 0]])
    p = IP.Pipe(d, "lineitem", LI, pool)
    key, qty, price = p.col("l_partkey"), p.col("l_quantity"), p.col("l_extendedprice")
    p.args = [key]
    pr = p.n("PROBE", 0, 0, 1, 1)
    brand, size, cont = p.n("PAYLOAD", pr, 1), p.n("PAYLOAD", pr, 2), p.n("PAYLOAD", pr, 3)
    arms = []
    for i, (br, lo) in enumerate((("Brand#12", 1), ("Brand#23", 10), ("Brand#34", 20))):
        lst = CONTAINERS[(i * 7) % len(CONTAINERS):] + CONTAINERS
        a = p.n("AND", p.n("EQ_CHAR", brand, p.cstr(br)), p.inlist(cont, lst[:n_containers], "right", "EQ_CHAR"))
        a = p.n("AND", a, p.n("AND", p.n("GE", qty, p.const(lo)), p.n("LE", qty, p.const(lo + 10))))
        a = p.n("AND", a, p.n("LE", size, p.const(5 * (i + 1))))
        arms.append(a)
    p.filter(p.n("OR", p.n("OR", arms[0], arms[1]), arms[2]))
    p.done(IP.SINK_AGG, [[price, 1, IP.SQL_BIGINT, 0], [0, 2, IP.SQL_BIGINT, 0]])
    return d


def test_q19_shape(engine, gpu_tabs, sf001):
    assert against_oracle(engine, gpu_tabs, sf001, q19_shape()) == 1


def test_in_build_pipeline(engine, gpu_tabs, sf001):
    d, pool = IP.new_plan({"orders": OR_, "lineitem": LI})
    b = IP.Pipe(d, "orders", OR_, pool)
    ok = b.col("o_orderkey")
    b.filter(b.inlist(b.col("o_orderpriority"), ["1-URGENT", "2-HIGH", "9-NONE", ""], "left", "EQ_CHAR"))
    b.filter(b.inlist(b.col("o_custkey"), int_consts(sf001["orders"]["o_custkey"], 300, 9)))
    b.done(IP.SINK_BUILD, [[ok, 0, IP.SQL_INT, 0], [b.col("o_totalprice"), 0, IP.SQL_BIGINT, 0]], keys=[[ok, 0, IP.SQL_INT, 0]])
    p = IP.Pipe(d, "lineitem", LI, pool)
    p.args = [p.col("l_orderkey")]
    pr = p.n("PROBE", 0, 0, 1, 1)
    tp = p.n("PAYLOAD", pr, 1)
    p.filter(p.inlist(p.col("l_linenumber"), [1, 3, 4], "right"))
    p.done(IP.SINK_AGG, [[tp, 1, IP.SQL_BIGINT, 0], [0, 2, IP.SQL_BIGINT, 0]], keys=[[p.col("l_returnflag"), 0, IP.SQL_CHAR, 1]])
    against_oracle(engine, gpu_tabs, sf001, d)
    engine.set_option("split_min_rows", 0)          # the same with the two-pass split forced
    engine.set_option("split_frac", 1e18)
    against_oracle(engine, gpu_tabs, sf001, d)


def test_in_nested_loops_condition(engine, gpu_tabs, sf001):
    d, pool = IP.new_plan({"orders": OR_, "lineitem": LI})
    a = IP.Pipe(d, "orders", OR_, pool)
    a.filter(a.n("LT", a.col("o_orderkey"), a.const(60)))
    a.done(IP.SINK_MAT, [[a.col("o_orderkey"), 0, IP.SQL_INT, 0], [a.col("o_custkey"), 0, IP.SQL_INT, 0]])
    b = IP.Pipe(d, "lineitem", LI, pool)
    b.filter(b.n("LT", b.col("l_orderkey"), b.const(40)))
    b.done(IP.SINK_MAT, [[b.col("l_partkey"), 0, IP.SQL_INT, 0], [b.col("l_linenumber"), 0, IP.SQL_INT, 0]])
    c = IP.Pipe(d, "lineitem", ["o_orderkey", "o_custkey", "l_partkey", "l_linenumber"], pool)
    c.filter(c.n("OR", c.inlist(c.n("ADD", c.n("COL", 1), c.n("COL", 3)), list(range(0, 3000, 7))),
                 c.inlist(c.n("COL", 0), [3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37, 41])))
    c.done(IP.SINK_AGG, [[c.n("COL", 2), 1, IP.SQL_BIGINT, 0], [0, 2, IP.SQL_BIGINT, 0]], source_kind=3, source_id=0)
    d["pipelines"][-1]["source_id2"] = 1
    assert against_oracle(engine, gpu_tabs, sf001, d) == 1


@pytest.mark.parametrize("group", [None, "l_linenumber", "l_returnflag"])
def test_register_aggregation(engine, gpu_tabs, sf001, group):
    consts = int_consts(sf001["lineitem"]["l_partkey"], 500, 2)
    assert agg_vs_numpy(engine, gpu_tabs, sf001, "lineitem", LI, "l_partkey", consts, "l_extendedprice", group) > 0


def test_late_materialized_select_star(engine, gpu_tabs, sf001):
    engine.set_option("late_materialize", 2)
    d = IP.select_in("lineitem", LI, "l_partkey", int_consts(sf001["lineitem"]["l_partkey"], 200, 8), [
        (c, IP.SQL_CHAR if c in ("l_shipmode", "l_shipinstruct") else IP.SQL_BIGINT, 25 if c.startswith("l_ship") and c != "l_shipdate" else 0)
        for c in LI if c not in ("l_returnflag",)])
    assert against_oracle(engine, gpu_tabs, sf001, d) > 0


def test_replay_and_graphs(engine, gpu_tabs, sf001):
    d = IP.select_in("lineitem", LI, "l_shipmode", ["MAIL", "SHIP", "AIR", "FOB", "RAIL", "TRUCK", "REG AIR"] * 2, OUT,
                     "right", "EQ_CHAR")
    d2 = IP.sum_in("lineitem", LI, "l_partkey", int_consts(sf001["lineitem"]["l_partkey"], 5000, 6), "l_extendedprice")
    for plan in (d, d2):
        first, _, _ = execute(engine, gpu_tabs, plan)
        for _ in range(4):
            again, _, tm = execute(engine, gpu_tabs, plan)
            assert sorted(again) == sorted(first)
        assert tm.host_syncs == 1


@pytest.mark.parametrize("k", [2, 5, 11])
def test_old_and_new_form_agree(engine, gpu_tabs, sf001, k):
    plans = [IP.select_in("lineitem", LI, "l_partkey", int_consts(sf001["lineitem"]["l_partkey"], k, k), OUT, "right"),
             IP.case_in("lineitem", LI, "l_shipmode", ["MAIL", "SHIP ", "AIR", "", "RAIL", "FOB", "X", "TRUCK", "Y", "Z", "W"][:k],
                        "l_quantity", eq="EQ_CHAR")]
    for d in plans:
        engine.set_option("in_lists", 0)
        old, _, _ = execute(engine, gpu_tabs, d)
        engine.set_option("in_lists", 2)
        new, _, _ = execute(engine, gpu_tabs, d)
        assert sorted(old) == sorted(new)


def test_internal_node_refused(engine, gpu_tabs):
    from resql_b200 import EngineError
    d = IP.select_in("lineitem", LI, "l_partkey", [1, 2, 3], OUT)
    d["pipelines"][0]["nodes"].append([1001, 0, 0, 0, 0])
    with pytest.raises(EngineError) as e:
        execute(engine, gpu_tabs, d)
    assert e.value.code == 1       # RQ_ERR_INVALID: the set node is internal to the library


@pytest.fixture(scope="module")
def fuzz_tabs(engine, sf001):
    from plan_fuzz import COLS
    up = {t: engine.upload(t, {c: sf001[t][c] for c, _ in cols}) for t, cols in COLS.items()}
    yield up
    for h in up.values():
        h.free()


@pytest.mark.parametrize("seed", range(250))
def test_random_plans_with_in_lists(seed, sf001, engine, fuzz_tabs):
    from resql_b200 import EngineError
    d = IP.random_inlist_plan(seed)
    tabs = plan_tables(d, sf001)
    try:
        want = serialize_columns(*run_plan(d, tabs))
    except ZeroDivisionError:
        pytest.skip("plan divides by zero")
    try:
        res, _ = engine.execute(Plan(d), {t["name"]: fuzz_tabs[t["name"]] for t in d["tables"]})
    except EngineError as e:
        if e.code == 3:
            pytest.fail(f"random plan {seed} is legal but was rejected: {e}")
        raise
    assert_same_relation(serialize_columns(res.columns, res.sql_types, res.sql_widths), want, d, f"random plan {seed}")


def test_sf1_partkey_list(engine):
    from resql_b200 import tpch
    L = tpch.generate(1, seed=3, tables=("lineitem",))["lineitem"]
    h = engine.upload("lineitem", {c: L[c] for c in LI})
    try:
        consts = int_consts(L["l_partkey"], 10000, 10)
        d = IP.sum_in("lineitem", LI, "l_partkey", consts, "l_extendedprice")
        res, _ = engine.execute(Plan(d), {"lineitem": h})
        m = np.isin(L["l_partkey"], np.array(consts))
        assert (int(res.columns[0][0]), int(res.columns[1][0])) == (int(L["l_extendedprice"][m].astype(np.int64).sum()), int(m.sum()))
    finally:
        h.free()
