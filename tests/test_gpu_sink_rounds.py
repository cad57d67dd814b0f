"""Sink rounds (engine_exec.inl "sink rounds"): a materialize whose computed outputs need more than the
12 value slots runs in the round variant of the scan kernel, which stores its values in rounds that
each fit the slots. Every result is checked against the plan oracle; the forced form (`sink_rounds` 2)
also runs plans the single sink holds, and must agree with it."""
import numpy as np
import pytest

from common import assert_same_relation, serialize_columns
from oracle.plan_oracle import run_plan
from resql_b200 import EngineError, Plan

from test_gpu_late_materialize import (ADD, BIGINT, BUILD, CONST, DIV, FILTER, LT, MUL, PAYLOAD, SUB, SRC_TABLE,
                                       Pipe, make_plan)

pytestmark = pytest.mark.gpu

RQ_ERR_UNSUPPORTED, RQ_ERR_RUNTIME = 3, 6


@pytest.fixture(scope="module")
def engine():
    from resql_b200 import Engine
    eng = Engine(0)
    yield eng
    eng.shutdown()


@pytest.fixture
def forced(engine):
    """rounds wherever they apply; every execution is lowered afresh (no replay of an earlier form)"""
    engine.set_option("sink_rounds", 2)
    engine.set_option("replay", 0)
    yield
    engine.set_option("sink_rounds", 1)
    engine.set_option("replay", 1)


def run(engine, d, tabs, handles=None):
    own = handles is None
    if own:
        handles = {n: engine.upload(n, c) for n, c in tabs.items()}
    try:
        res, tm = engine.execute(Plan(d), handles)
    finally:
        if own:
            for h in handles.values():
                h.free()
    return serialize_columns(res.columns, res.sql_types, res.sql_widths), tm


def check(engine, d, tabs, what=""):
    got, tm = run(engine, d, tabs)
    assert_same_relation(got, serialize_columns(*run_plan(d, tabs)), d, what)
    return got


def table(n, seed):
    rng = np.random.default_rng(seed)
    return {"t": {"k": rng.permutation(n).astype(np.int64),
                  "v": rng.integers(-(1 << 40), 1 << 40, n, dtype=np.int64),
                  "d": rng.integers(0, 1000, n, dtype=np.int64).astype(np.int32)}}


def computed_select(m, shared=False, filt=None, divisor=None):
    """select k + 0, v + 1, v + 2, ... (m outputs, all computed) from t [where d < filt]; `shared`: every
    output also reads one common product v * 3, which stays live across the rounds"""
    p = Pipe(SRC_TABLE, 0)
    k, v, dd = p.col(0), p.col(1), p.col(2)
    if filt is not None:
        p.filt(p.n(LT, dd, p.const(filt)))
    base = p.n(MUL, v, p.const(3)) if shared else v
    p.val(p.n(ADD, k, p.const(0)))
    for j in range(1, m):
        x = p.n(ADD, base, p.const(j))
        if j % 3 == 0:
            x = p.n(SUB, x, dd)
        p.val(x)
    if divisor is not None:          # the last output divides by (d - divisor): zero for some rows
        p.d["vals"][-1][0] = p.n(DIV, v, p.n(SUB, dd, p.const(divisor)))
    return make_plan([("t", ["k", "v", "d"])], [p])


@pytest.mark.parametrize("m", [13, 24, 64])
@pytest.mark.parametrize("n", [0, 1, 255, 256, 257, 300_001])
def test_computed_select_list(m, n, engine):
    tabs = table(n, seed=m * 7 + n)
    check(engine, computed_select(m, filt=700), tabs, f"{m} outputs, {n} rows")


@pytest.mark.parametrize("m", [13, 24, 64])
def test_computed_select_list_order_by_limit(m, engine):
    tabs = table(20_000, seed=m)
    d = computed_select(m, shared=True)
    d["order"], d["limit"] = [[m - 1, 1], [0, 0]], 25
    check(engine, d, tabs, f"{m} outputs, order by limit")


@pytest.mark.parametrize("m", [5, 13, 40])
def test_forced_rounds_match_the_oracle(m, engine, forced):
    tabs = table(50_000, seed=100 + m)
    check(engine, computed_select(m, shared=True, filt=500), tabs, f"{m} outputs, forced rounds")


def test_division_by_zero_in_a_late_round(engine):
    tabs = table(10_000, seed=5)
    with pytest.raises(EngineError) as e:
        run(engine, computed_select(30, divisor=17), tabs)
    assert e.value.code == RQ_ERR_RUNTIME
    tabs["t"]["d"][:] = 5                    # no zero divisor: the same plan runs
    check(engine, computed_select(30, divisor=17), tabs, "division")


def join_plus_computed(tabs, m):
    """select pt.*, bt.* (payloads), and m computed outputs over both sides: the late form defers the
    plain columns and its record pipeline takes the rounds"""
    bt, pt = tabs["bt"], tabs["pt"]
    b = Pipe(SRC_TABLE, 0, sink=BUILD)
    bn = [b.col(i) for i in range(len(bt))]
    b.key(bn[0])
    for nd in bn:
        b.val(nd)
    p = Pipe(SRC_TABLE, 1)
    pn = [p.col(i) for i in range(len(pt))]
    pr = p.probe(0, [pn[0]], single=1)
    pays = [p.n(PAYLOAD, pr, j) for j in range(len(bt))]
    for nd in pn + pays:
        p.val(nd)
    for j in range(m):
        p.val(p.n(ADD, p.n(MUL, pn[1 + j % 3], p.const(j + 2)), pays[1 + j % 2]))
    return make_plan([("bt", list(bt)), ("pt", list(pt))], [b, p])


@pytest.mark.parametrize("m", [13, 30])
def test_select_star_over_a_join_plus_computed(m, engine):
    rng = np.random.default_rng(m)
    nb, npr = 5000, 200_000
    tabs = {"bt": {"bk": rng.permutation(nb).astype(np.int64),
                   **{f"b{c}": rng.integers(-1000, 1000, nb, dtype=np.int64) for c in range(4)}},
            "pt": {"pk": rng.integers(0, 2 * nb, npr, dtype=np.int64),
                   **{f"p{c}": rng.integers(-1000, 1000, npr, dtype=np.int64) for c in range(4)}}}
    check(engine, join_plus_computed(tabs, m), tabs, f"join + {m} computed")


def test_replay_and_graph_executions(engine):
    tabs = table(100_000, seed=9)
    d = computed_select(40, shared=True, filt=900)
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
        assert sorted(got) == sorted(runs[0][0])       # (a materialize's row order is unspecified)
    assert runs[-1][1].host_syncs == 1


def random_wide_plan(seed):
    """13 to 40 outputs, each a random expression over the three columns and up to 5 shared
    sub-expressions. Each output starts with a constant of its own, so the plan's CSE shares no more of
    it with other outputs: the shared sub-expressions are what stays live across rounds. Every such plan
    must run (the test fails on any refusal)."""
    rng = np.random.default_rng(seed)
    p = Pipe(SRC_TABLE, 0)
    leaves = [p.col(0), p.col(1), p.col(2)]
    if rng.random() < 0.5:
        p.filt(p.n(LT, leaves[2], p.const(int(rng.integers(100, 1000)))))
    pool = list(leaves)
    for _ in range(int(rng.integers(0, 6))):          # shared sub-expressions
        pool.append(p.n(int(rng.choice([ADD, SUB, MUL])), int(rng.choice(pool)), p.const(int(rng.integers(-50, 50)))))
    m = int(rng.integers(13, 41))          # (at most 3 units an output: the program stays within 128 units)
    for j in range(m):
        x = p.n(int(rng.choice([ADD, SUB, MUL])), int(rng.choice(pool)), p.const(100_000 + j))
        for _ in range(int(rng.integers(0, 3))):
            y = int(rng.choice(pool)) if rng.random() < 0.5 else p.const(int(rng.integers(-1000, 1000)))
            x = p.n(int(rng.choice([ADD, SUB, MUL])), x, y)
        p.val(x)
    return make_plan([("t", ["k", "v", "d"])], [p])


@pytest.mark.parametrize("seed", range(50))
def test_random_wide_select_lists(seed, engine):
    tabs = table(int(np.random.default_rng(seed).integers(1, 30_000)), seed=1000 + seed)
    check(engine, random_wide_plan(seed), tabs, f"seed {seed}")
