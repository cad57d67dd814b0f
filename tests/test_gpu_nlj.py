"""Nested-loops joins (RQ_SRC_CROSS) streamed through the scan kernel: the pairs of the two child
relations are staged tile by tile and never materialized. Small cases are checked against the plan
oracle; large ones (up to 4.9e9 pairs) against a numpy evaluation that never builds the product:
one side sorted, searchsorted, then prefix sums (exact int64 with wrap-around, like the engine)."""
import random

import numpy as np
import pytest

from common import serialize_columns, assert_same_relation
from oracle.plan_oracle import run_plan
from resql_b200 import Plan

pytestmark = pytest.mark.gpu

COL, CONST, ADD, SUB, MUL, DIV = 1, 2, 4, 5, 6, 7
LT, LE, GT, GE, EQ, NEQ, EQ_CHAR = 10, 11, 12, 13, 14, 15, 16
FILTER, PROBE, PAYLOAD = 22, 23, 24
SUM, COUNT, MIN, MAX = 1, 2, 3, 4
CHAR, BIGINT = 1, 4
SRC_TABLE, SRC_PIPE, SRC_CROSS = 1, 2, 3
AGG, BUILD, MAT = 1, 2, 3
RQ_ERR_UNSUPPORTED, RQ_ERR_RUNTIME = 3, 6
M64 = (1 << 64) - 1


@pytest.fixture(scope="module")
def engine():
    from resql_b200 import Engine
    eng = Engine(0)
    yield eng
    eng.shutdown()


class Pipe:
    def __init__(self, kind, sid, sid2=0, sink=MAT, size_hint=0):
        self.d = {"source_kind": kind, "source_id": sid, "source_id2": sid2, "sink_kind": sink,
                  "size_hint": size_hint, "nodes": [], "args": [], "keys": [], "vals": []}

    def n(self, op, a=0, b=0, c=0, imm=0):
        self.d["nodes"].append([op, a, b, c, imm])
        return len(self.d["nodes"]) - 1

    def col(self, i):
        return self.n(COL, i)

    def const(self, v):
        return self.n(CONST, imm=int(v))

    def filt(self, cond):
        self.n(FILTER, cond)

    def key(self, node, sql=BIGINT, w=0):
        self.d["keys"].append([node, 0, sql, w])

    def val(self, node, kind=0, sql=BIGINT, w=0):
        self.d["vals"].append([node, kind, sql, w])


def child(tid, cols, sql=None, lt=None):
    """materializes columns `cols` of table `tid`, optionally where column 0 < lt"""
    p = Pipe(SRC_TABLE, tid)
    nodes = [p.col(c) for c in cols]
    if lt is not None:
        p.filt(p.n(LT, nodes[0], p.const(lt)))
    for k, nd in enumerate(nodes):
        s, w = (sql[k] if sql else (BIGINT, 0))
        p.val(nd, 0, s, w)
    return p


def plan(tables, pipes, order=(), strpool=""):
    last = pipes[-1].d
    n_out = len(last["keys"]) + len(last["vals"])
    return {"tables": [{"name": n, "columns": list(c)} for n, c in tables], "pipelines": [p.d for p in pipes],
            "order": [list(o) for o in order], "limit": -1, "strpool": strpool,
            "result_names": [f"c{i}" for i in range(n_out)], "result_types": ["BIGINT"] * n_out}


def run(engine, d, tabs):
    handles = {n: engine.upload(n, c) for n, c in tabs.items()}
    try:
        res, tm = engine.execute(Plan(d), handles)
    finally:
        for h in handles.values():
            h.free()
    return res, tm


def check_oracle(engine, d, tabs, what=""):
    res, tm = run(engine, d, tabs)
    got = serialize_columns(res.columns, res.sql_types, res.sql_widths)
    want = serialize_columns(*run_plan(d, tabs))
    assert_same_relation(got, want, d, what)
    return got, tm


def tables(nl, nr, ncols=2, seed=0, lo=-1000, hi=1000):
    rng = np.random.default_rng(seed)
    mk = lambda n, p: {f"{p}{c}": rng.integers(lo, hi, n, dtype=np.int64) for c in range(ncols)}
    return {"l": mk(nl, "a"), "r": mk(nr, "b")}


def names(tabs):
    return [(n, list(c.keys())) for n, c in tabs.items()]


# ---- sizes around tile and side boundaries --------------------------------------------------------
SIZES = [0, 1, 63, 255, 256, 257, 1025]


@pytest.mark.parametrize("nl", SIZES)
@pytest.mark.parametrize("nr", SIZES)
def test_boundary_sizes_count_sum_and_emit(nl, nr, engine):
    """COUNT / SUM over both sides under l.a0 < r.b0, and the selective pairs themselves; nr < 64
    puts many outer rows into one tile"""
    tabs = tables(nl, nr, seed=nl * 7919 + nr)
    agg = Pipe(SRC_CROSS, 0, 1, AGG)
    a0, a1, b0, b1 = (agg.col(i) for i in range(4))
    agg.filt(agg.n(LT, a0, b0))
    agg.val(a0, COUNT)
    agg.val(agg.n(ADD, a1, b1), SUM)
    check_oracle(engine, plan(names(tabs), [child(0, [0, 1]), child(1, [0, 1]), agg]), tabs, f"agg {nl}x{nr}")
    emit = Pipe(SRC_CROSS, 0, 1, MAT)
    a0, a1, b0, b1 = (emit.col(i) for i in range(4))
    emit.filt(emit.n(LT, emit.n(ADD, a0, b0), emit.const(-1500)))
    for nd in (a1, b1, a0, b0):
        emit.val(nd)
    check_oracle(engine, plan(names(tabs), [child(0, [0, 1]), child(1, [0, 1]), emit]), tabs, f"emit {nl}x{nr}")


# ---- numpy evaluation of  SELECT count(*), sum(l.x), sum(r.y), min(r.y), max(l.x) WHERE l.a < r.b ----
def reference_lt(la, lx, rb, ry):
    """exact, without the product: for each left row the right rows with b > a are a suffix of r
    sorted by b"""
    o = np.argsort(rb, kind="stable")
    bs, ys = rb[o], ry[o].astype(np.uint64)
    suf_sum = np.concatenate([np.cumsum(ys[::-1], dtype=np.uint64)[::-1], np.zeros(1, np.uint64)])
    suf_min = np.concatenate([np.minimum.accumulate(ry[o][::-1])[::-1], [np.iinfo(np.int64).max]])
    first = np.searchsorted(bs, la, side="right")       # first right row with b > a
    cnt = (len(rb) - first).astype(np.int64)
    count = int(cnt.sum())
    sum_x = int((lx.astype(np.uint64) * cnt.astype(np.uint64)).sum(dtype=np.uint64))
    sum_y = int(suf_sum[first].sum(dtype=np.uint64))
    min_y = int(suf_min[first].min()) if count else None
    max_x = int(lx[cnt > 0].max()) if count else None
    s64 = lambda v: v - (1 << 64) if v >= (1 << 63) else v
    return count, s64(sum_x & M64), s64(sum_y & M64), min_y, max_x


def lt_agg_plan(tabs, kinds=(COUNT, SUM, SUM, MIN, MAX)):
    p = Pipe(SRC_CROSS, 0, 1, AGG)
    la, lx, rb, ry = (p.col(i) for i in range(4))
    p.filt(p.n(LT, la, rb))
    nodes = [la, lx, ry, ry, lx]
    for k, nd in zip(kinds, nodes):
        p.val(nd, k)
    return plan(names(tabs), [child(0, [0, 1]), child(1, [0, 1]), p])


@pytest.mark.parametrize("nl,nr,full", [(20_000, 20_000, True), (70_000, 70_000, False)])
def test_beyond_the_old_materialization_limit(nl, nr, full, engine):
    """4e8 pairs (COUNT, SUM, MIN, MAX) and 4.9e9 pairs (more than 2^32: pair indices need 64 bits)"""
    rng = np.random.default_rng(nl)
    big = np.int64(1) << 62
    tabs = {"l": {"a0": rng.integers(0, 1 << 30, nl, dtype=np.int64), "a1": rng.integers(-big, big, nl, dtype=np.int64)},
            "r": {"b0": rng.integers(0, 1 << 30, nr, dtype=np.int64), "b1": rng.integers(-big, big, nr, dtype=np.int64)}}
    kinds = (COUNT, SUM, SUM, MIN, MAX) if full else (COUNT, SUM, SUM)
    res, tm = run(engine, lt_agg_plan(tabs, kinds), tabs)
    want = reference_lt(tabs["l"]["a0"], tabs["l"]["a1"], tabs["r"]["b0"], tabs["r"]["b1"])
    got = tuple(int(c[0]) for c in res.columns)
    assert got == want[:len(kinds)]
    assert want[0] > (1 << 31 if not full else 1 << 27)      # (the count itself does not fit 31 bits)


@pytest.mark.parametrize("n", [1 << 20, 1_050_000])
def test_pair_limit_is_refused_before_the_join_runs(n, engine):
    """2^40 pairs and more: RQ_ERR_UNSUPPORTED naming the limit, raised before the join's launch. The
    join, had it been launched, would stream 1.1e12 pairs (seconds at 1.2e11 pairs/s); the refused
    execution and a small one queued behind it on the same stream finish far sooner."""
    import time
    from resql_b200 import EngineError
    tabs = {"l": {"a0": np.arange(n, dtype=np.int64)}, "r": {"b0": np.arange(n, dtype=np.int64)}}
    p = Pipe(SRC_CROSS, 0, 1, AGG)
    p.filt(p.n(LT, p.col(0), p.col(1)))
    p.val(0, COUNT)
    small = Pipe(SRC_TABLE, 0, sink=AGG)
    small.val(small.col(0), SUM)
    handles = {k: engine.upload(k, c) for k, c in tabs.items()}
    try:
        t0 = time.perf_counter()
        with pytest.raises(EngineError) as e:
            engine.execute(Plan(plan(names(tabs), [child(0, [0]), child(1, [0]), p])), handles)
        res, _ = engine.execute(Plan(plan(names(tabs), [small])), handles)
        elapsed = time.perf_counter() - t0
    finally:
        for h in handles.values():
            h.free()
    assert e.value.code == RQ_ERR_UNSUPPORTED and "nested-loops join" in str(e.value) and "2^40" in str(e.value)
    assert int(res.columns[0][0]) == n * (n - 1) // 2
    assert elapsed < 3.0, f"{elapsed:.2f} s: the refused join seems to have run"


def test_many_groups_beyond_2_to_the_32_pairs(engine):
    """GROUP BY with 1000 groups (hash aggregation) over 4.9e9 pairs: the first hash table is sized
    from a bounded guess, not from the pair count"""
    nl = nr = 70_000
    rng = np.random.default_rng(17)
    big = np.int64(1) << 62
    tabs = {"l": {"a0": rng.integers(0, 1 << 30, nl, dtype=np.int64), "a1": np.arange(nl, dtype=np.int64) % 1000},
            "r": {"b0": rng.integers(0, 1 << 30, nr, dtype=np.int64), "b1": rng.integers(-big, big, nr, dtype=np.int64)}}
    p = Pipe(SRC_CROSS, 0, 1, AGG)
    la, lg, rb, ry = (p.col(i) for i in range(4))
    p.filt(p.n(LT, la, rb))
    p.key(lg)
    p.val(la, COUNT); p.val(ry, SUM)
    res, _ = run(engine, plan(names(tabs), [child(0, [0, 1]), child(1, [0, 1]), p]), tabs)
    # per left row: count and wrap-around sum of the right rows with b > a (a suffix of r sorted by b)
    o = np.argsort(tabs["r"]["b0"], kind="stable")
    bs, ys = tabs["r"]["b0"][o], tabs["r"]["b1"][o].astype(np.uint64)
    suf = np.concatenate([np.cumsum(ys[::-1], dtype=np.uint64)[::-1], np.zeros(1, np.uint64)])
    first = np.searchsorted(bs, tabs["l"]["a0"], side="right")
    cnt = nr - first
    g = tabs["l"]["a1"]
    want_cnt = np.zeros(1000, np.int64); np.add.at(want_cnt, g, cnt)
    want_sum = np.zeros(1000, np.uint64); np.add.at(want_sum, g, suf[first])
    want = {k: (int(want_cnt[k]), int(want_sum[k].astype(np.int64))) for k in range(1000) if want_cnt[k]}
    got = {int(k): (int(c), int(s)) for k, c, s in zip(*res.columns)}
    assert int(want_cnt.sum()) > 1 << 31
    assert got == want


# ---- every sink over a cross source ---------------------------------------------------------------
def test_emit_regrows_past_the_first_capacity(engine):
    """the first output capacity is the input size capped at 2^24 rows; 8000 x 8000 pairs of which
    about 32e6 survive make the materialize regrow its output once"""
    tabs = tables(8000, 8000, seed=3, lo=0, hi=10_000)
    p = Pipe(SRC_CROSS, 0, 1, MAT)
    a0, a1, b0, b1 = (p.col(i) for i in range(4))
    p.filt(p.n(LT, a0, b0))
    p.val(a1); p.val(b1)
    d = plan(names(tabs), [child(0, [0, 1]), child(1, [0, 1]), p])
    res, tm = run(engine, d, tabs)
    la, lx, rb, ry = tabs["l"]["a0"], tabs["l"]["a1"], tabs["r"]["b0"], tabs["r"]["b1"]
    want = reference_lt(la, lx, rb, ry)
    assert len(res.columns[0]) == want[0] > (1 << 24)
    assert int(res.columns[0].astype(np.uint64).sum(dtype=np.uint64)) == want[1] & M64
    assert int(res.columns[1].astype(np.uint64).sum(dtype=np.uint64)) == want[2] & M64


def test_lowagg_with_group_keys_from_both_sides(engine):
    tabs = tables(700, 900, seed=5)
    tabs["l"]["a2"] = (np.arange(700) % 3).astype(np.int64)
    tabs["r"]["b2"] = (np.arange(900) % 2).astype(np.int64)
    p = Pipe(SRC_CROSS, 0, 1, AGG)
    a0, a1, a2, b0, b1, b2 = (p.col(i) for i in range(6))
    p.filt(p.n(GT, p.n(SUB, a0, b0), p.const(100)))
    p.key(a2); p.key(b2)
    p.val(a0, COUNT); p.val(b1, SUM); p.val(a1, MIN); p.val(p.n(MUL, a1, b1), MAX)
    check_oracle(engine, plan(names(tabs), [child(0, [0, 1, 2]), child(1, [0, 1, 2]), p]), tabs, "lowagg")


def test_hashagg_with_many_groups(engine):
    """about 20 000 groups: the hash aggregation"""
    tabs = tables(200, 5000, seed=6)
    tabs["l"]["a2"] = np.arange(200, dtype=np.int64)
    tabs["r"]["b2"] = np.arange(5000, dtype=np.int64) % 100
    p = Pipe(SRC_CROSS, 0, 1, AGG)
    a0, a1, a2, b0, b1, b2 = (p.col(i) for i in range(6))
    p.filt(p.n(LE, a0, b0))
    p.key(a2); p.key(b2)
    p.val(a0, COUNT); p.val(p.n(ADD, a1, b1), SUM)
    got, _ = check_oracle(engine, plan(names(tabs), [child(0, [0, 1, 2]), child(1, [0, 1, 2]), p]), tabs, "hashagg")
    assert len(got) > 15_000


def _nlj_then_probe(tabs, single):
    """NLJ result (l.a0, r.b1 where l.a0 < r.b0) is the build side of a join with table p on key"""
    nlj = Pipe(SRC_CROSS, 0, 1, BUILD)
    a0, a1, b0, b1 = (nlj.col(i) for i in range(4))
    nlj.filt(nlj.n(LT, a0, b0))
    nlj.key(a1); nlj.val(b1)
    probe = Pipe(SRC_TABLE, 2, sink=AGG)
    k, v = probe.col(0), probe.col(1)
    probe.d["args"] = [k]
    pr = probe.n(PROBE, 2, 0, 1, 1 if single else 0)
    pay = probe.n(PAYLOAD, pr, 0)
    probe.val(k, COUNT); probe.val(probe.n(ADD, v, pay), SUM); probe.val(pay, MIN)
    return plan(names(tabs), [child(0, [0, 1]), child(1, [0, 1]), nlj, probe])


@pytest.mark.parametrize("unique", [True, False])
def test_build_side_of_a_later_hash_join(unique, engine):
    tabs = tables(40, 300, seed=7)
    if unique:      # one pair per key: l.a1 distinct and exactly one right row passes for each
        tabs["l"]["a1"] = np.arange(40, dtype=np.int64) * 3
        tabs["r"]["b0"] = np.full(300, -10_000, dtype=np.int64)
        tabs["r"]["b0"][0] = 10_000
    tabs["p"] = {"k": np.arange(-2000, 2000, dtype=np.int64), "v": np.arange(4000, dtype=np.int64)}
    check_oracle(engine, _nlj_then_probe(tabs, unique), tabs, "nlj build")


@pytest.mark.parametrize("single", [True, False])
def test_probe_inside_the_nlj_pipeline(single, engine):
    """single-match probe, and a multi-match one (duplicate build keys: the expansion pass A reads
    the cross source)"""
    tabs = tables(150, 200, seed=8)
    n = 64 if single else 256
    tabs["p"] = {"k": (np.arange(n) % 64).astype(np.int64) - 32, "v": np.arange(n, dtype=np.int64) * 1000}
    build = Pipe(SRC_TABLE, 2, sink=BUILD)
    k, v = build.col(0), build.col(1)
    build.key(k); build.val(v)
    p = Pipe(SRC_CROSS, 1, 2, MAT)
    a0, a1, b0, b1 = (p.col(i) for i in range(4))
    p.filt(p.n(LT, a0, b0))
    key = p.n(SUB, a1, b1)
    p.d["args"] = [p.n(DIV, key, p.const(50))]
    pr = p.n(PROBE, 0, 0, 1, 1 if single else 0)
    pay = p.n(PAYLOAD, pr, 0)
    p.val(a0); p.val(b1); p.val(pay)
    d = plan([("p", ["k", "v"]), ("l", ["a0", "a1"]), ("r", ["b0", "b1"])],
             [build, child(1, [0, 1]), child(2, [0, 1]), p])
    check_oracle(engine, d, tabs, f"probe single={single}")


# ---- other conditions -----------------------------------------------------------------------------
def test_strings_from_both_sides(engine):
    rng = np.random.default_rng(9)
    seg = np.array([b"AUTO", b"BUILDING", b"MACHINERY"], dtype="S11")
    tabs = {"l": {"a0": rng.integers(0, 100, 300, dtype=np.int64), "s": seg[rng.integers(0, 3, 300)]},
            "r": {"b0": rng.integers(0, 100, 200, dtype=np.int64), "t": seg[rng.integers(0, 3, 200)]}}
    sql = [(BIGINT, 0), (CHAR, 10)]
    p = Pipe(SRC_CROSS, 0, 1, MAT)
    a0, s, b0, t = (p.col(i) for i in range(4))
    p.filt(p.n(EQ_CHAR, s, t))
    p.filt(p.n(LT, a0, b0))
    p.val(s, 0, CHAR, 10); p.val(t, 0, CHAR, 10); p.val(a0)
    check_oracle(engine, plan(names(tabs), [child(0, [0, 1], sql), child(1, [0, 1], sql), p]), tabs, "strings")
    g = Pipe(SRC_CROSS, 0, 1, AGG)
    a0, s, b0, t = (g.col(i) for i in range(4))
    g.filt(g.n(NEQ, a0, b0))
    g.key(s, CHAR, 10); g.key(t, CHAR, 10)
    g.val(a0, COUNT); g.val(b0, SUM)
    check_oracle(engine, plan(names(tabs), [child(0, [0, 1], sql), child(1, [0, 1], sql), g]), tabs, "string keys")


def test_avg_over_pairs(engine):
    """AVG as the planner lowers it: SUM and COUNT, then their quotient in a pipeline over the result"""
    tabs = tables(400, 500, seed=10)
    g = Pipe(SRC_CROSS, 0, 1, AGG)
    a0, a1, b0, b1 = (g.col(i) for i in range(4))
    g.filt(g.n(GE, a0, b0))
    g.val(g.n(SUB, a1, b1), SUM); g.val(a0, COUNT)
    f = Pipe(SRC_PIPE, 2)
    s, c = f.col(0), f.col(1)
    f.val(f.n(DIV, f.n(MUL, s, f.const(100)), c)); f.val(c)
    check_oracle(engine, plan(names(tabs), [child(0, [0, 1]), child(1, [0, 1]), g, f]), tabs, "avg")


def test_division_by_zero_in_the_condition_is_reported(engine):
    from resql_b200 import EngineError
    tabs = tables(300, 300, seed=11)
    tabs["r"]["b1"][123] = 0
    p = Pipe(SRC_CROSS, 0, 1, AGG)
    a0, a1, b0, b1 = (p.col(i) for i in range(4))
    p.filt(p.n(GT, p.n(DIV, a0, b1), p.const(0)))
    p.val(a0, COUNT)
    with pytest.raises(EngineError) as e:
        run(engine, plan(names(tabs), [child(0, [0, 1]), child(1, [0, 1]), p]), tabs)
    assert e.value.code == RQ_ERR_RUNTIME


def test_wide_children_stage_only_what_the_pipeline_reads(engine):
    """9 + 9 child columns, 4 of them read: only those are staged"""
    tabs = tables(300, 400, ncols=9, seed=12)
    p = Pipe(SRC_CROSS, 0, 1, AGG)
    a3, a7, b2, b8 = p.col(3), p.col(7), p.col(9 + 2), p.col(9 + 8)
    p.filt(p.n(LT, p.n(ADD, a3, b2), p.n(SUB, a7, b8)))
    p.val(a3, COUNT); p.val(p.n(MUL, a7, b8), SUM); p.val(b2, MAX)
    check_oracle(engine, plan(names(tabs), [child(0, list(range(9))), child(1, list(range(9))), p]), tabs, "wide")


# ---- repeated execution -----------------------------------------------------------------------------
def test_careful_replay_and_graph_runs_are_identical(engine):
    tabs = tables(3000, 2000, seed=13)
    emit = Pipe(SRC_CROSS, 0, 1, MAT)
    a0, a1, b0, b1 = (emit.col(i) for i in range(4))
    emit.filt(emit.n(LT, emit.n(ADD, a0, b0), emit.const(-1700)))
    emit.val(a1); emit.val(b1)
    d = plan(names(tabs), [child(0, [0, 1], lt=500), child(1, [0, 1]), emit])
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
        assert_same_relation(got, want, d, "nlj repeated")
    assert runs[-1][1].host_syncs == 1, f"replay waited {runs[-1][1].host_syncs} times"


# ---- random plans -----------------------------------------------------------------------------------
def _random_case(seed):
    rng = random.Random(seed)
    sink = rng.choice([MAT, AGG, AGG, BUILD])
    nl = rng.choice([0, 1, 5, 63, 200, 700, 1000])
    nr = rng.choice([0, 1, 3, 64, 255] + ([] if sink == MAT else [600, 1000]))     # (oracle time: rows out)
    tabs = tables(nl, nr, ncols=3, seed=seed, lo=-rng.choice([10, 1000, 1 << 40]), hi=rng.choice([10, 1000, 1 << 40]))
    kids = [child(t, [0, 1, 2], lt=rng.choice([None, 0, 500])) for t in (0, 1)]
    p = Pipe(SRC_CROSS, 0, 1, AGG if sink == BUILD else sink)
    c = [p.col(i) for i in range(6)]
    L, R = c[:3], c[3:]

    def side_expr(cols):
        x = rng.choice(cols)
        if rng.random() < 0.5:
            x = p.n(rng.choice([ADD, SUB, MUL]), x, rng.choice(cols + [p.const(rng.randint(-5, 5))]))
        return x
    cond = p.n(rng.choice([LT, LE, GT, GE, EQ, NEQ]), side_expr(L), side_expr(R))
    if rng.random() < 0.3:
        cond = p.n(rng.choice([8, 9]), cond, p.n(rng.choice([LT, GT]), rng.choice(L + R), p.const(rng.randint(-500, 500))))
    p.filt(cond)
    pipes = kids + [p]
    if sink == MAT:
        for _ in range(rng.randint(1, 4)):
            p.val(side_expr(rng.choice([L, R, L + R])))
    elif sink == AGG:
        for _ in range(rng.randint(0, 2)):
            k = rng.choice(L + R)
            p.key(p.n(SUB, k, p.n(MUL, p.n(DIV, k, p.const(7)), p.const(7))) if rng.random() < 0.5 else k)
        for _ in range(rng.randint(1, 4)):
            p.val(side_expr(L + R), rng.choice([SUM, COUNT, MIN, MAX]))
    else:       # the NLJ as a join build, probed by the left child again
        p.d["sink_kind"] = BUILD
        p.key(rng.choice(L)); p.val(side_expr(R))
        q = Pipe(SRC_PIPE, 0, sink=AGG)
        k = q.col(0)
        q.d["args"] = [k]
        pr = q.n(PROBE, 2, 0, 1, 0)
        q.val(k, COUNT); q.val(q.n(PAYLOAD, pr, 0), SUM)
        pipes.append(q)
    return plan(names(tabs), pipes), tabs


@pytest.mark.parametrize("seed", range(100))
def test_random_nlj_plans_match_oracle(seed, engine):
    d, tabs = _random_case(seed)
    check_oracle(engine, d, tabs, f"seed {seed}")
