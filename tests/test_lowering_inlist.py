"""CPU check of the IN-list set unit: OR trees of equality tests against constants are lowered to one
H_INSET unit (rq_debug_lower prints the unit and its set decoded from the device form), and the program
run by the VM models with the set test (tests/vm_model_inset.py: host units and encoded device program)
reproduces the plan oracle."""
import numpy as np
import pytest

from common import serialize_columns, assert_same_relation
from oracle import plan_oracle as PO
from resql_b200 import native as N
from resql_b200.plan import Plan
import inlist_plans as IP
import vm_model_inset as vm_model

LI = ["l_orderkey", "l_partkey", "l_linenumber", "l_quantity", "l_extendedprice", "l_returnflag", "l_shipmode",
      "l_shipinstruct"]
OUT = [("l_orderkey", IP.SQL_INT, 0), ("l_extendedprice", IP.SQL_BIGINT, 0)]


@pytest.fixture(scope="module")
def li(sf001):
    return {c: np.asarray(sf001["lineitem"][c])[:6000] for c in LI}


@pytest.fixture(autouse=True)
def default_in_lists():
    yield
    N.load().rq_set_option(b"in_lists", 1.0)


def set_in_lists(v):
    assert N.load().rq_set_option(b"in_lists", float(v)) == 0


def lower(d):
    types, widths = [], []
    for c in d["tables"][0]["columns"]:
        t, w = vm_model.phys_of(np.zeros(1, dtype=_dtype[c]))
        types.append(t); widths.append(w)
    return N.debug_lower(Plan(d), 0, vm_model.IMPL_EMIT, types, widths)


_dtype = {"l_orderkey": np.int32, "l_partkey": np.int32, "l_linenumber": np.int32, "l_quantity": np.int64,
          "l_extendedprice": np.int64, "l_returnflag": np.uint8, "l_shipmode": "S11", "l_shipinstruct": "S26"}


def check(d, li, level, expect_units=None):
    """runs pipeline 0 of d over li in the VM model at `level` and compares with the oracle"""
    tabs = {"lineitem": {c: li[c] for c in d["tables"][0]["columns"]}}
    src = [np.asarray(tabs["lineitem"][c]) for c in d["tables"][0]["columns"]]
    pool = d["strpool"].encode("latin1")
    pool_strings = {nd[4]: pool[nd[4]:].split(b"\0")[0] for nd in d["pipelines"][0]["nodes"] if nd[0] == 3}
    run = vm_model.run_pipeline_vm if level == "host" else vm_model.run_pipeline_device
    out = run(Plan(d), 0, src, pool_strings, vm_model.IMPL_REGAGG)
    last = d["pipelines"][-1]
    st = [k[2] for k in last["keys"]] + [v[2] for v in last["vals"]]
    sw = [k[3] for k in last["keys"]] + [v[3] for v in last["vals"]]
    got = serialize_columns(*PO.finish(d, out, st, sw))
    want = serialize_columns(*PO.run_plan(d, tabs))
    assert_same_relation(got, want, d, "in list")
    if expect_units is not None:
        units = [l for l in vm_model_units(d)]
        assert sum(1 for u in units if u[0] == vm_model.H_INSET) == expect_units
    return len(want)


def vm_model_units(d):
    return vm_model.parse(lower(d))["unit"]


def _consts(li, col, k, seed, extra=()):
    rng = np.random.default_rng(seed)
    vals = np.unique(li[col])
    pick = list(rng.choice(vals, size=min(k, len(vals)), replace=False)) if k else []
    while len(pick) < k:
        pick.append(int(rng.integers(-1000, 10 ** 7)))
    return [int(x) for x in pick] + list(extra)


@pytest.mark.parametrize("level", ["host", "device"])
@pytest.mark.parametrize("shape", ["right", "left", "balanced"])
@pytest.mark.parametrize("k", [1, 2, 11, 12, 65, 1000])
def test_integer_lists_all_shapes(li, k, shape, level):
    consts = _consts(li, "l_partkey", k, k)
    d = IP.select_in("lineitem", LI, "l_partkey", consts, OUT, shape)
    rows = check(d, li, level, expect_units=1 if k >= 2 else 0)
    assert k < 11 or rows > 0


@pytest.mark.parametrize("level", ["host", "device"])
@pytest.mark.parametrize("col,k", [("l_linenumber", 3), ("l_orderkey", 40), ("l_quantity", 12), ("l_returnflag", 2),
                                   ("l_extendedprice", 65)])
def test_column_widths(li, col, k, level):
    consts = _consts(li, col, k, 7)
    d = IP.select_in("lineitem", LI, col, consts, OUT, "right", const_left=(k % 2 == 0))
    check(d, li, level, expect_units=1)


@pytest.mark.parametrize("level", ["host", "device"])
def test_computed_operand(li, level):
    d = IP.select_in("lineitem", LI, "l_linenumber", [2, 4, 6, 8], OUT, "left", computed=True)
    check(d, li, level, expect_units=1)


@pytest.mark.parametrize("level", ["host", "device"])
def test_duplicate_and_out_of_range_constants(li, level):
    # duplicates make CSE share leaves between ORs of the tree; constants outside the column's values
    # (and outside int32) are dropped or can never match
    consts = [3, 5, 3, 3, 7, 5, -1, 0, 2 ** 31, -(2 ** 40), 1, 1]
    for col in ("l_linenumber", "l_orderkey", "l_returnflag"):
        d = IP.select_in("lineitem", LI, col, consts, OUT, "right")
        check(d, li, level, expect_units=1)


@pytest.mark.parametrize("level", ["host", "device"])
@pytest.mark.parametrize("eq,col", [("EQ_CHAR", "l_shipmode"), ("EQ_VARCHAR", "l_shipmode"), ("EQ_CHAR", "l_shipinstruct"),
                                    ("EQ_VARCHAR", "l_shipinstruct")])
def test_string_lists(li, eq, col, level):
    consts = ["MAIL", "AIR  ", "REG AIR", "", "TRUCK     XX", "TRUCK", "SHIP", "SHIP", "NONE ", "DELIVER IN PERSON",
              "TAKE BACK RETURN AND MORE THAN THE COLUMN", "COLLECT COD"]
    d = IP.select_in("lineitem", LI, col, consts, OUT, "right", eq)
    check(d, li, level, expect_units=1)


@pytest.mark.parametrize("level", ["host", "device"])
def test_thousand_strings(li, level):
    consts = [f"S{i:05d}" + "x" * (i % 7) for i in range(998)] + ["RAIL", "FOB"]
    d = IP.select_in("lineitem", LI, "l_shipmode", consts, OUT, "balanced", "EQ_CHAR")
    assert check(d, li, level, expect_units=1) > 0


@pytest.mark.parametrize("level", ["host", "device"])
def test_in_list_inside_case(li, level):
    d = IP.case_in("lineitem", LI, "l_linenumber", [1, 3, 5, 7], "l_extendedprice")
    check(d, li, level, expect_units=1)
    d = IP.case_in("lineitem", LI, "l_shipmode", ["MAIL", "SHIP", "AIR", "FOB"], "l_quantity", eq="EQ_CHAR")
    check(d, li, level, expect_units=1)


@pytest.mark.parametrize("level", ["host", "device"])
def test_two_lists_ored(li, level):
    d = IP.two_lists("lineitem", LI, "l_linenumber", [1, 2, 3], "l_partkey", _consts(li, "l_partkey", 30, 3), OUT)
    check(d, li, level, expect_units=2)


def test_aggregate_over_in_list(li):
    d = IP.sum_in("lineitem", LI, "l_partkey", _consts(li, "l_partkey", 50, 5), "l_extendedprice", group="l_linenumber")
    check(d, li, "device", expect_units=1)


def test_in_lists_option(li):
    # in_lists 0 is the unrolled lowering: the 12-value right-deep list needs more than 12 live values
    consts = _consts(li, "l_partkey", 12, 12)
    d = IP.select_in("lineitem", LI, "l_partkey", consts, OUT, "right")
    set_in_lists(0)
    with pytest.raises(N.EngineError, match="live temporaries"):
        lower(d)
    small = IP.select_in("lineitem", LI, "l_partkey", consts[:5], OUT, "right")
    assert not any(u[0] == vm_model.H_INSET for u in vm_model_units(small))
    check(small, li, "device")
    set_in_lists(2)
    assert any(u[0] == vm_model.H_INSET for u in vm_model_units(small))
    check(small, li, "device")
    set_in_lists(1)
    check(d, li, "device", expect_units=1)


def test_long_list_lowers_as_one_unit():
    # 10^5 values: recognition, dead-code elimination and filter hoisting see one node
    consts = list(range(0, 300000, 3))
    d = IP.select_in("lineitem", LI, "l_partkey", consts, OUT, "right")
    prog = vm_model.parse(lower(d))
    assert [u[0] for u in prog["unit"]] == [vm_model.H_INSET]
    (form, mem), = prog["sets"].values()
    assert form == vm_model.IS_BITMAP and len(mem) == len(consts)
    # x IN (...) AND y > 3: the AND split under FILTER must not walk the OR chain recursively
    d, pool = IP.new_plan({"lineitem": LI})
    p = IP.Pipe(d, "lineitem", LI, pool)
    p.filter(p.n("AND", p.inlist(p.col("l_partkey"), consts, "left"), p.n("GT", p.col("l_linenumber"), p.const(3))))
    p.done(IP.SINK_MAT, [[p.col("l_orderkey"), 0, IP.SQL_INT, 0]])
    assert sum(1 for u in vm_model.parse(lower(d))["unit"] if u[0] == vm_model.H_INSET) == 1


def test_set_forms():
    # a dense list is a bitmap, a sparse one a sorted array
    dense = vm_model.parse(lower(IP.select_in("lineitem", LI, "l_partkey", list(range(100, 200)), OUT)))["sets"]
    sparse = vm_model.parse(lower(IP.select_in("lineitem", LI, "l_partkey", [i * 100003 for i in range(64)], OUT)))["sets"]
    assert [f for f, _ in dense.values()] == [vm_model.IS_BITMAP]
    assert [f for f, _ in sparse.values()] == [vm_model.IS_SORTED]


@pytest.mark.parametrize("seed", range(40))
def test_random_plans_with_in_lists(seed, sf001):
    """random single-table plans with injected lists through both VM levels"""
    d = IP.random_inlist_plan(seed)
    if len(d["pipelines"]) != 1 or d["pipelines"][0]["sink_kind"] == 2:
        pytest.skip("multi-pipeline plans run on the GPU (test_gpu_inlist.py)")
    t = d["tables"][d["pipelines"][0]["source_id"]]
    tabs = {t["name"]: {c: np.asarray(sf001[t["name"]][c])[:5000] for c in t["columns"]}}
    src = [tabs[t["name"]][c] for c in t["columns"]]
    pool = d["strpool"].encode("latin1")
    pool_strings = {nd[4]: pool[nd[4]:].split(b"\0")[0] for nd in d["pipelines"][0]["nodes"] if nd[0] == 3}
    try:
        want = serialize_columns(*PO.run_plan(d, tabs))
    except ZeroDivisionError:
        pytest.skip("plan divides by zero")
    last = d["pipelines"][-1]
    st = [k[2] for k in last["keys"]] + [v[2] for v in last["vals"]]
    sw = [k[3] for k in last["keys"]] + [v[3] for v in last["vals"]]
    for run in (vm_model.run_pipeline_vm, vm_model.run_pipeline_device):
        out = run(Plan(d), 0, src, pool_strings, vm_model.IMPL_REGAGG)
        assert_same_relation(serialize_columns(*PO.finish(d, out, st, sw)), want, d, f"random plan {seed}")
