"""Late materialization (IMPL_LATE, engine_exec.inl "late materialization"): materialize pipelines
wider than the early form holds (more than 24 outputs, 16 staged columns, 12 live values or 8
string columns) run as a record of references written by the scan plus one gather launch. Every
result is checked against the plan oracle (or the golden outputs of the fixtures); with
`late_materialize` 2 the late form also runs every plan it applies to, so both paths are compared
on the same plans."""
import numpy as np
import pytest

from common import (assert_same_relation, load_golden, load_plan_dict, plan_names, plan_tables,
                    serialize_columns)
from oracle.plan_oracle import run_plan
from resql_b200 import EngineError, Plan, tpch

pytestmark = pytest.mark.gpu

COL, CONST, ADD, SUB, MUL, DIV = 1, 2, 4, 5, 6, 7
LT, LE, GT, GE, EQ = 10, 11, 12, 13, 14
FILTER, PROBE, PAYLOAD = 22, 23, 24
SUM, COUNT, MIN, MAX = 1, 2, 3, 4
VARCHAR, CHAR, INT, BIGINT = 0, 1, 3, 4
SRC_TABLE, SRC_PIPE, SRC_CROSS = 1, 2, 3
AGG, BUILD, MAT = 1, 2, 3
RQ_ERR_UNSUPPORTED, RQ_ERR_RUNTIME = 3, 6


@pytest.fixture(scope="module")
def engine():
    from resql_b200 import Engine
    eng = Engine(0)
    yield eng
    eng.shutdown()


@pytest.fixture
def late_first(engine):
    engine.set_option("late_materialize", 2)
    yield
    engine.set_option("late_materialize", 1)


class Pipe:
    def __init__(self, kind, sid, sid2=0, sink=MAT):
        self.d = {"source_kind": kind, "source_id": sid, "source_id2": sid2, "sink_kind": sink,
                  "size_hint": 0, "nodes": [], "args": [], "keys": [], "vals": []}

    def n(self, op, a=0, b=0, c=0, imm=0):
        self.d["nodes"].append([op, a, b, c, imm])
        return len(self.d["nodes"]) - 1

    def col(self, i):
        return self.n(COL, i)

    def const(self, v):
        return self.n(CONST, imm=int(v))

    def filt(self, cond):
        self.n(FILTER, cond)

    def probe(self, build, keys, single=0):
        b = len(self.d["args"])
        self.d["args"].extend(keys)
        return self.n(PROBE, build, b, len(keys), single)

    def key(self, node, st=(BIGINT, 0)):
        self.d["keys"].append([node, 0, st[0], st[1]])

    def val(self, node, st=(BIGINT, 0), kind=0):
        self.d["vals"].append([node, kind, st[0], st[1]])


def make_plan(tables, pipes, order=(), limit=-1):
    last = pipes[-1].d
    n_out = len(last["keys"]) + len(last["vals"])
    return {"tables": [{"name": n, "columns": list(c)} for n, c in tables], "pipelines": [p.d for p in pipes],
            "order": [list(o) for o in order], "limit": limit, "strpool": "",
            "result_names": [f"c{i}" for i in range(n_out)], "result_types": ["BIGINT"] * n_out}


def execute(engine, d, handles):
    return engine.execute(Plan(d), handles)


def check(engine, d, tabs, handles=None, what=""):
    own = handles is None
    if own:
        handles = {n: engine.upload(n, c) for n, c in tabs.items()}
    try:
        res, tm = execute(engine, d, handles)
    finally:
        if own:
            for h in handles.values():
                h.free()
    got = serialize_columns(res.columns, res.sql_types, res.sql_widths)
    want = serialize_columns(*run_plan(d, tabs))
    assert_same_relation(got, want, d, what)
    return got, tm


# ---- synthetic wide tables -----------------------------------------------------------------------
STR_WIDTHS = (2, 5, 12, 26)


def wide_table(ncols, n, seed):
    """column 0: a permutation of 0..n-1 (filters keep an exact number of rows); then I32, I8, I64 and
    strings of several widths in turn (more than 8 string columns from 17 columns up)"""
    rng = np.random.default_rng(seed)
    cols, sql = {"k": rng.permutation(n).astype(np.int64)}, [(BIGINT, 0)]
    for c in range(1, ncols):
        kind = c % 4
        if kind == 0:
            cols[f"c{c}"] = rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64); sql.append((BIGINT, 0))
        elif kind == 1:
            cols[f"c{c}"] = rng.integers(-(1 << 31), (1 << 31) - 1, n, dtype=np.int64).astype(np.int32); sql.append((INT, 0))
        elif kind == 2 and c % 8 == 2:
            cols[f"c{c}"] = rng.integers(65, 91, n, dtype=np.int64).astype(np.uint8); sql.append((CHAR, 1))
        else:
            w = STR_WIDTHS[c % len(STR_WIDTHS)]
            letters = rng.integers(97, 123, (n, w), dtype=np.int64).astype(np.uint8)
            lens = rng.integers(0, w + 1, n)
            letters[np.arange(w)[None, :] >= lens[:, None]] = 0
            arr = np.zeros((n, w + 1), np.uint8)
            arr[:, :w] = letters
            cols[f"c{c}"] = arr.view(f"S{w + 1}").reshape(n)
            sql.append((VARCHAR if c % 3 else CHAR, w))
    return cols, sql


FILTERS = {"all": None, "none": ("lt", 0), "one": ("eq", 0), "pct": ("lt", None)}


def select_star(ncols, sql, n, filt):
    p = Pipe(SRC_TABLE, 0)
    nodes = [p.col(c) for c in range(ncols)]
    f = FILTERS[filt]
    if f is not None:
        k = f[1] if f[1] is not None else max(n // 100, 1)
        p.filt(p.n(LT if f[0] == "lt" else EQ, nodes[0], p.const(k)))
    for c in range(ncols):
        p.val(nodes[c], sql[c])
    return p


SIZES = [0, 1, 255, 256, 257, 1023, 1025, 300_001]


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("ncols", [17, 40, 64])
def test_wide_select_star_owned(ncols, n, engine):
    tabs_cols, sql = wide_table(ncols, n, seed=ncols * 1000 + n)
    tabs = {"w": tabs_cols}
    handles = {"w": engine.upload("w", tabs_cols)}
    try:
        for filt in FILTERS:
            d = make_plan([("w", list(tabs_cols))], [select_star(ncols, sql, n, filt)])
            _, tm = check(engine, d, tabs, handles, f"{ncols} cols, {n} rows, {filt}")
    finally:
        handles["w"].free()


@pytest.mark.parametrize("n", [1, 257, 1025, 300_001])
@pytest.mark.parametrize("ncols", [17, 64])
def test_wide_select_star_borrowed(ncols, n, engine):
    """device columns used in place (no padding: the gather never reads past n_rows)"""
    import torch
    from resql_b200.native import RQ_I8, RQ_I32, RQ_I64, RQ_STR
    tabs_cols, sql = wide_table(ncols, n, seed=ncols + n)
    keep, dev = [], {}
    for name, a in tabs_cols.items():
        raw = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
        t = torch.from_numpy(raw.copy()).cuda()
        keep.append(t)
        ty = {np.dtype(np.int64): (RQ_I64, 8), np.dtype(np.int32): (RQ_I32, 4), np.dtype(np.uint8): (RQ_I8, 1)}.get(a.dtype)
        if ty is None:
            ty = (RQ_STR, a.dtype.itemsize)
        dev[name] = (t.data_ptr(), ty[0], ty[1])
    torch.cuda.synchronize()
    h = engine.upload_device("w", dev, n)
    try:
        for filt in ("all", "pct", "one"):
            d = make_plan([("w", list(tabs_cols))], [select_star(ncols, sql, n, filt)])
            check(engine, d, {"w": tabs_cols}, {"w": h}, f"borrowed {ncols} cols, {n} rows, {filt}")
    finally:
        h.free()
        del keep


# ---- joins over TPC-H data -------------------------------------------------------------------------
def schema(t):
    return [(c, tpch.sql_type_of(k, a)) for c, k, a in tpch.SCHEMAS[t]]


def build_all(tid, t, key_col):
    """build over every column of table t, keyed on key_col"""
    sc = schema(t)
    b = Pipe(SRC_TABLE, tid, sink=BUILD)
    nodes = [b.col(i) for i in range(len(sc))]
    b.key(nodes[key_col], sc[key_col][1])
    for i, (_, st) in enumerate(sc):
        b.val(nodes[i], st)
    return b


@pytest.fixture(scope="module")
def tp():
    return tpch.generate(0.05, seed=3, tables=("lineitem", "orders", "customer"))


def tp_tabs(tp, names):
    return {t: {c: tp[t][c] for c, _ in schema(t)} for t in names}


def lineitem_orders(filters=()):
    """select * from lineitem, orders where l_orderkey = o_orderkey [and filters on lineitem]: 25 columns"""
    lsc, osc = schema("lineitem"), schema("orders")
    p = Pipe(SRC_TABLE, 1)
    ln = [p.col(i) for i in range(len(lsc))]
    for op, c, k in filters:
        p.filt(p.n(op, ln[c], p.const(k)))
    pr = p.probe(0, [ln[0]], single=1)
    pays = [p.n(PAYLOAD, pr, j) for j in range(len(osc))]
    for i, (_, st) in enumerate(lsc):
        p.val(ln[i], st)
    for j, (_, st) in enumerate(osc):
        p.val(pays[j], st)
    return make_plan([("orders", [c for c, _ in osc]), ("lineitem", [c for c, _ in lsc])], [build_all(0, "orders", 0), p])


@pytest.mark.parametrize("direct", [1, 0])
def test_lineitem_orders_select_star(direct, tp, engine):
    engine.set_option("direct_joins", direct)
    try:
        got, tm = check(engine, lineitem_orders(), tp_tabs(tp, ("orders", "lineitem")), what=f"l x o direct={direct}")
        assert len(got) == len(tp["lineitem"]["l_orderkey"])
        assert len(got[0].split("|")) == 26
    finally:
        engine.set_option("direct_joins", 1)


def test_zone_skipped_selection_keeps_absolute_row_ids(tp, engine):
    """a range on the sorted l_orderkey restricts the scan to a tile range: the record's row ids are
    absolute rows of lineitem"""
    lk = np.sort(tp["lineitem"]["l_orderkey"])
    assert len(lk) >= 1 << 18
    lo, hi = int(lk[len(lk) // 3]), int(lk[len(lk) // 3 + 5000])
    d = lineitem_orders([(GE, 0, lo), (LE, 0, hi)])
    got, _ = check(engine, d, tp_tabs(tp, ("orders", "lineitem")), what="zone skipped")
    assert 5000 <= len(got) < 6000


def customer_orders_lineitem(extra_filter=None):
    """select * from customer, orders, lineitem where c_custkey = o_custkey and o_orderkey = l_orderkey:
    33 columns; the lineitem pipeline carries 17 payloads of one probe"""
    csc, osc, lsc = schema("customer"), schema("orders"), schema("lineitem")
    bc = build_all(0, "customer", 0)
    po = Pipe(SRC_TABLE, 1, sink=BUILD)
    on = [po.col(i) for i in range(len(osc))]
    pr = po.probe(0, [on[1]], single=1)
    cp = [po.n(PAYLOAD, pr, j) for j in range(len(csc))]
    po.key(on[0], osc[0][1])
    for j, (_, st) in enumerate(csc):
        po.val(cp[j], st)
    for i, (_, st) in enumerate(osc):
        po.val(on[i], st)
    pl = Pipe(SRC_TABLE, 2)
    ln = [pl.col(i) for i in range(len(lsc))]
    if extra_filter:
        pl.filt(pl.n(LT, ln[extra_filter[0]], pl.const(extra_filter[1])))
    pr2 = pl.probe(1, [ln[0]], single=1)
    pays = [pl.n(PAYLOAD, pr2, j) for j in range(len(csc) + len(osc))]
    for j, (_, st) in enumerate(csc + osc):
        pl.val(pays[j], st)
    for i, (_, st) in enumerate(lsc):
        pl.val(ln[i], st)
    return make_plan([("customer", [c for c, _ in csc]), ("orders", [c for c, _ in osc]),
                      ("lineitem", [c for c, _ in lsc])], [bc, po, pl])


def test_customer_orders_lineitem_select_star(tp, engine):
    got, _ = check(engine, customer_orders_lineitem(), tp_tabs(tp, ("customer", "orders", "lineitem")), what="c x o x l")
    assert len(got[0].split("|")) == 34


def dup_tables(n_build, n_probe, ncols, seed):
    rng = np.random.default_rng(seed)
    b = {"bk": rng.integers(0, 50, n_build, dtype=np.int64)}
    p = {"pk": rng.integers(0, 60, n_probe, dtype=np.int64)}
    for c in range(ncols):
        b[f"b{c}"] = rng.integers(-1000, 1000, n_build, dtype=np.int64)
        p[f"p{c}"] = rng.integers(-1000, 1000, n_probe, dtype=np.int64)
    return {"bt": b, "pt": p}


def many_to_many(tabs, divide=False):
    """wide join with duplicate keys on both sides (one row per match), and a computed output that
    uses a payload of the multi-match probe"""
    bt, pt = tabs["bt"], tabs["pt"]
    b = Pipe(SRC_TABLE, 0, sink=BUILD)
    bn = [b.col(i) for i in range(len(bt))]
    b.key(bn[0])
    for nd in bn:
        b.val(nd)
    p = Pipe(SRC_TABLE, 1)
    pn = [p.col(i) for i in range(len(pt))]
    pr = p.probe(0, [pn[0]])
    pays = [p.n(PAYLOAD, pr, j) for j in range(len(bt))]
    for nd in pn + pays:
        p.val(nd)
    p.val(p.n(DIV if divide else ADD, pn[1], pays[1]))
    return make_plan([("bt", list(bt)), ("pt", list(pt))], [b, p])


def test_many_to_many_wide_join(engine):
    tabs = dup_tables(400, 3000, 13, seed=5)        # 2 x 14 + 1 = 29 outputs
    got, _ = check(engine, many_to_many(tabs), tabs, what="many-to-many")
    assert len(got) > 3000


def test_many_to_many_forced_late_matches_early(engine, late_first):
    tabs = dup_tables(300, 2000, 5, seed=6)         # 13 outputs: the early form holds it too
    check(engine, many_to_many(tabs), tabs, what="many-to-many, late first")


def test_division_by_zero_in_a_computed_output(engine):
    tabs = dup_tables(100, 500, 13, seed=7)
    tabs["bt"]["b0"][:] = 0
    with pytest.raises(EngineError) as e:
        check(engine, many_to_many(tabs, divide=True), tabs)
    assert e.value.code == RQ_ERR_RUNTIME


# ---- nested-loops join -----------------------------------------------------------------------------
def child(tid, ncols):
    p = Pipe(SRC_TABLE, tid)
    for c in range(ncols):
        p.val(p.col(c))
    return p


def wide_nlj(nl, nr, ncols, seed, margin):
    rng = np.random.default_rng(seed)
    tabs = {"l": {f"a{c}": rng.integers(0, 1 << 20, nl, dtype=np.int64) for c in range(ncols)},
            "r": {f"b{c}": rng.integers(0, 1 << 20, nr, dtype=np.int64) for c in range(ncols)}}
    p = Pipe(SRC_CROSS, 0, 1)
    nodes = [p.col(i) for i in range(2 * ncols)]
    p.filt(p.n(LT, p.n(ADD, nodes[0], p.const(margin)), nodes[ncols]))
    for nd in nodes:
        p.val(nd)
    return tabs, make_plan([("l", list(tabs["l"])), ("r", list(tabs["r"]))], [child(0, ncols), child(1, ncols), p])


def test_wide_nlj_select_star(engine):
    tabs, d = wide_nlj(1025, 1023, 13, seed=1, margin=0)       # 26 outputs, about half the pairs
    check(engine, d, tabs, what="wide NLJ")


def test_wide_nlj_selective_4e8_pairs(engine):
    """20000 x 20000 pairs, a condition few pairs pass; checked against numpy without the product"""
    tabs, d = wide_nlj(20_000, 20_000, 13, seed=2, margin=(1 << 20) - 3000)
    handles = {n: engine.upload(n, c) for n, c in tabs.items()}
    try:
        res, _ = execute(engine, d, handles)
    finally:
        for h in handles.values():
            h.free()
    la, rb = tabs["l"]["a0"], tabs["r"]["b0"]
    margin = (1 << 20) - 3000
    o = np.argsort(rb, kind="stable")
    want = []
    for i in np.nonzero(la + margin < rb.max())[0]:
        for j in o[np.searchsorted(rb[o], la[i] + margin, side="right"):]:
            want.append(tuple(int(tabs["l"][f"a{c}"][i]) for c in range(13)) + tuple(int(tabs["r"][f"b{c}"][j]) for c in range(13)))
    got = list(zip(*[[int(v) for v in c] for c in res.columns]))
    assert sorted(got) == sorted(want) and len(want) > 0


# ---- downstream of a wide result -------------------------------------------------------------------
@pytest.mark.parametrize("order,limit", [([(5, 0), (0, 1), (3, 1)], 10), ([(5, 1), (0, 1), (3, 1)], -1)])
def test_order_by_over_a_wide_result(order, limit, tp, engine):
    d = lineitem_orders([(LT, 0, 2000)])
    d["order"], d["limit"] = [list(o) for o in order], limit
    check(engine, d, tp_tabs(tp, ("orders", "lineitem")), what="order by")


def test_large_full_order_by_over_a_wide_result(tp, engine):
    d = lineitem_orders()
    d["order"] = [[16 + 4, 1], [0, 1], [3, 1]]        # o_orderdate, l_orderkey, l_linenumber
    check(engine, d, tp_tabs(tp, ("orders", "lineitem")), what="large order by")


def test_aggregation_over_a_33_column_intermediate(tp, engine):
    d = customer_orders_lineitem()
    agg = Pipe(SRC_PIPE, 2, sink=AGG)
    mseg, qty, price, okey = agg.col(6), agg.col(8 + 9 + 4), agg.col(8 + 9 + 5), agg.col(8)
    agg.key(mseg, (CHAR, 10))
    agg.val(qty, kind=SUM)
    agg.val(price, kind=MAX)
    agg.val(okey, kind=COUNT)
    d["pipelines"].append(agg.d)
    d["result_names"] = ["a", "b", "c", "d"]
    d["result_types"] = ["BIGINT"] * 4
    check(engine, d, tp_tabs(tp, ("customer", "orders", "lineitem")), what="agg over 33 columns")


# ---- both paths on the same plans ------------------------------------------------------------------
@pytest.mark.parametrize("name", plan_names())
def test_fixtures_with_late_first(name, sf001, engine):
    d = load_plan_dict(name)
    tabs = plan_tables(d, sf001)
    handles = {n: engine.upload(n, c) for n, c in tabs.items()}
    try:
        # each form twice: the second run starts from what the first one learned (expansion, sizes)
        res1, _ = execute(engine, d, handles)
        res1, tm1 = execute(engine, d, handles)
        engine.set_option("late_materialize", 2)
        try:
            res2, _ = execute(engine, d, handles)
            res2, tm2 = execute(engine, d, handles)
        finally:
            engine.set_option("late_materialize", 1)
    finally:
        for h in handles.values():
            h.free()
    _, want = load_golden(name)
    for res in (res1, res2):
        assert_same_relation(serialize_columns(res.columns, res.sql_types, res.sql_widths), want, d, name)
    late = any(p["sink_kind"] == MAT and any(d["pipelines"][p_i]["nodes"][v[0]][0] in (COL, PAYLOAD) for v in p["vals"])
               for p_i, p in enumerate(d["pipelines"]) if p["source_kind"] in (SRC_TABLE, SRC_PIPE, SRC_CROSS))
    if late:
        assert tm2.kernel_launches > tm1.kernel_launches, f"{name}: the late form did not run"


@pytest.mark.parametrize("seed", range(250))
def test_random_plans_with_late_first(seed, sf001, engine, late_first):
    from plan_fuzz import random_plan
    d = random_plan(seed)
    tabs = plan_tables(d, sf001)
    try:
        want = serialize_columns(*run_plan(d, tabs))
    except ZeroDivisionError:
        pytest.skip("plan divides by zero")
    handles = {n: engine.upload(n, c) for n, c in tabs.items()}
    try:
        res, _ = execute(engine, d, handles)
    finally:
        for h in handles.values():
            h.free()
    assert_same_relation(serialize_columns(res.columns, res.sql_types, res.sql_widths), want, d, f"seed {seed}")


# ---- repeated execution ----------------------------------------------------------------------------
def test_repeated_execution_of_a_wide_join(tp, engine):
    d = lineitem_orders([(LT, 10, 9000)])
    tabs = tp_tabs(tp, ("orders", "lineitem"))
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
        assert_same_relation(got, want, d, "repeated")
        assert got == runs[0][0]
    assert runs[-1][1].host_syncs == 1


# ---- refusals --------------------------------------------------------------------------------------
def test_65_output_columns_are_refused_before_any_launch(engine):
    cols, sql = wide_table(65, 100, seed=1)
    big = {"k": np.arange(1 << 22, dtype=np.int64)}
    agg = Pipe(SRC_TABLE, 1, sink=AGG)
    agg.val(agg.col(0), kind=SUM)
    wide = select_star(65, sql, 100, "all")
    wide.d["source_id"] = 0
    d = make_plan([("w", list(cols)), ("big", ["k"])], [agg, wide])
    handles = {"w": engine.upload("w", cols), "big": engine.upload("big", big)}
    try:
        with pytest.raises(EngineError) as e:
            execute(engine, d, handles)
    finally:
        for h in handles.values():
            h.free()
    assert e.value.code == RQ_ERR_UNSUPPORTED and "64" in str(e.value)


def test_build_with_more_than_24_payloads_keeps_its_error(engine):
    cols, sql = wide_table(30, 100, seed=2)
    b = Pipe(SRC_TABLE, 0, sink=BUILD)
    nodes = [b.col(i) for i in range(30)]
    b.key(nodes[0])
    for i in range(30):
        b.val(nodes[i], sql[i])
    p = Pipe(SRC_TABLE, 0)
    pr = p.probe(0, [p.col(0)], single=1)
    for i in range(30):
        p.val(p.n(PAYLOAD, pr, i), sql[i])
    d = make_plan([("w", list(cols))], [b, p])
    h = engine.upload("w", cols)
    try:
        with pytest.raises(EngineError) as e:
            execute(engine, d, {"w": h})
    finally:
        h.free()
    assert e.value.code == RQ_ERR_UNSUPPORTED
