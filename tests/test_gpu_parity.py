"""GPU parity tests proper: every plan fixture (lowered by the host shim from the reference's own
planner output) is executed through the C ABI on the B200 and must reproduce (a) the output of
the reference engine itself (tests/golden/sf001/*.out) and (b) the oracle, bit for bit."""
import os
import subprocess

import numpy as np
import pytest

from common import (ROOT, plan_names, load_plan_dict, load_golden, plan_tables, serialize_columns,
                    assert_same_relation)
from oracle.plan_oracle import run_plan
from resql_b200 import Plan, tpch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from resql_b200 import Engine
    eng = Engine(0)
    yield eng
    eng.shutdown()


def _run(engine, d, tabs):
    handles = {n: engine.upload(n, c) for n, c in tabs.items()}
    try:
        res, tm = engine.execute(Plan(d), handles)
    finally:
        for h in handles.values():
            h.free()
    return serialize_columns(res.columns, res.sql_types, res.sql_widths), tm


@pytest.mark.parametrize("name", plan_names())
def test_fixture_matches_reference_engine(name, sf001, engine):
    d = load_plan_dict(name)
    got, tm = _run(engine, d, plan_tables(d, sf001))
    _, want = load_golden(name)
    assert_same_relation(got, want, d, name)
    assert tm.kernel_launches > 0


@pytest.mark.parametrize("name", ["q1", "q6", "agg_linenumber", "agg_wrap", "agg_nogroup_minmax", "case_sum"])
@pytest.mark.parametrize("rows", [0, 1, 255, 256, 257, 1023, 1024, 1025, 5000, 300_001])
def test_ragged_sizes_match_oracle(name, rows, engine):
    """empty, single-row, tile-boundary and multi-CTA inputs (tile = 256 tuples)"""
    d = load_plan_dict(name)
    data = tpch.generate(0.06, seed=1234, tables=("lineitem",))
    tabs = plan_tables(d, data)
    tabs = {n: {c: v[:rows] for c, v in cols.items()} for n, cols in tabs.items()}
    got, _ = _run(engine, d, tabs)
    want = serialize_columns(*run_plan(d, tabs))
    assert_same_relation(got, want, d, f"{name}@{rows}")


def test_sf1_q1_q6_match_oracle(engine):
    """BASELINE config[1]: SF1 Q1/Q6 on one B200, bit-exact against the oracle"""
    data = tpch.generate(1.0, seed=99, tables=("lineitem",))
    for name in ("q1", "q6"):
        d = load_plan_dict(name)
        tabs = plan_tables(d, data)
        got, tm = _run(engine, d, tabs)
        want = serialize_columns(*run_plan(d, tabs))
        assert_same_relation(got, want, d, name + "@sf1")


@pytest.mark.parametrize("case", ["fits", "outliers", "narrow_off"])
def test_transfer_narrowing_is_exact(case, engine):
    """Uploads from host buffers send 8-byte columns over PCIe in 1 or 4 bytes when every value fits and
    widen them again on the device (host_narrow.h); the width is GUESSED from a sample. Values the sample
    cannot see (a single wide or negative value at an unsampled row) must widen the transfer, not be
    truncated: results stay identical to the oracle, and to the engine with narrowing switched off."""
    data = tpch.generate(0.4, seed=4321, tables=("lineitem",))
    li = data["lineitem"]
    n = len(li["l_quantity"])
    assert n >= 4 * 512 * 1024
    if case == "outliers":
        li["l_quantity"] = li["l_quantity"].copy(); li["l_quantity"][n // 2 + 1] = 300            # no longer one byte
        li["l_discount"] = li["l_discount"].copy(); li["l_discount"][7] = -3                      # negative: not a byte
        li["l_extendedprice"] = li["l_extendedprice"].copy(); li["l_extendedprice"][n - 5] = 1 << 33   # not int32
        li["l_tax"] = li["l_tax"].copy(); li["l_tax"][n // 3 + 2] = -(1 << 40)
        li["l_linenumber"] = li["l_linenumber"].copy(); li["l_linenumber"][n // 5 + 3] = 300     # INT column: no longer one byte
    if case == "narrow_off":
        engine.set_option("narrow", 0)
    try:
        for name in ("q1", "q6", "agg_nogroup_minmax", "agg_wrap", "agg_linenumber"):
            d = load_plan_dict(name)
            tabs = plan_tables(d, data)
            if name == "agg_linenumber":          # (an INT column whose values fit one byte: 1..7, or 300 in the outlier case)
                assert "l_linenumber" in tabs["lineitem"]
            got, _ = _run(engine, d, tabs)
            want = serialize_columns(*run_plan(d, tabs))
            assert_same_relation(got, want, d, f"{name} ({case})")
    finally:
        engine.set_option("narrow", 1)


def _range_plan(filters):
    """select count(*), sum(v), min(k), max(k) from t where <filters on k>; filters = [(op, const)]"""
    nodes = [[1, 0, 0, 0, 0], [1, 1, 0, 0, 0]]
    for op, c in filters:
        nodes.append([2, 0, 0, 0, int(c)])
        nodes.append([op, 0, len(nodes) - 1, 0, 0])
        nodes.append([22, len(nodes) - 1, 0, 0, 0])
    return {"tables": [{"name": "t", "columns": ["k", "v"]}],
            "pipelines": [{"source_kind": 1, "source_id": 0, "source_id2": 0, "sink_kind": 1, "size_hint": 0, "nodes": nodes, "args": [],
                           "keys": [], "vals": [[0, 2, 4, 0], [1, 1, 4, 0], [0, 3, 4, 0], [0, 4, 4, 0]]},
                          {"source_kind": 2, "source_id": 0, "source_id2": 0, "sink_kind": 3, "size_hint": 0,
                           "nodes": [[1, 0, 0, 0, 0], [1, 1, 0, 0, 0], [1, 2, 0, 0, 0], [1, 3, 0, 0, 0]], "args": [], "keys": [],
                           "vals": [[0, 0, 4, 0], [1, 0, 4, 0], [2, 0, 4, 0], [3, 0, 4, 0]]}],
            "order": [], "limit": -1, "strpool": "", "result_names": ["n", "s", "lo", "hi"], "result_types": ["BIGINT"] * 4}


@pytest.mark.parametrize("dtype", ["int64", "int32"])
def test_zone_skipping_on_sorted_columns_is_exact(dtype, engine):
    """A selection on a column whose values are non-decreasing over the rows restricts the scan to a
    tile range (engine_exec.inl "tile ranges"); the result must be the one of the full scan. Keys with
    duplicates and gaps, ranges that start / end inside tiles, empty and out-of-domain ranges."""
    import numpy as np
    rng = np.random.default_rng(11)
    n = 1_500_003
    k = np.cumsum(rng.integers(0, 3, n)).astype(dtype) + 1000            # sorted, duplicates, gaps
    v = rng.integers(-10**9, 10**9, n).astype(np.int64)
    t = {"t": {"k": k, "v": v}}
    LT, LE, GT, GE, EQ = 10, 11, 12, 13, 14
    lo, hi, mid = int(k[0]), int(k[-1]), int(k[n // 2])
    cases = [[(GE, mid), (LE, mid + 5000)], [(GT, mid), (LT, mid + 3)], [(EQ, int(k[777_777]))], [(EQ, mid), (EQ, mid + 1)],
             [(GE, lo), (LE, hi)], [(GT, hi)], [(LT, lo)], [(LE, lo)], [(GE, hi)], [(GE, hi + 10)], [(LE, lo - 10)],
             [(GE, int(k[255])), (LE, int(k[256]))], [(GE, int(k[n - 300]))], [(LE, int(k[300]))], [(GT, -2**31), (LT, 2**31 - 1)]]
    for zs in (1, 0):
        engine.set_option("zone_skip", zs)
        try:
            h = engine.upload("t", t["t"])
            for f in cases:
                d = _range_plan(f)
                res, _ = engine.execute(Plan(d), {"t": h})
                got = serialize_columns(res.columns, res.sql_types, res.sql_widths)
                want = serialize_columns(*run_plan(d, t))
                assert got == want, f"filters {f} zone_skip={zs}: {got} != {want}"
            h.free()
        finally:
            engine.set_option("zone_skip", 1)


def test_char_equality_has_comparechar_semantics(engine):
    """compareChar (qlib/scalar.h:27-46) on a CHAR column against constants: equality ignores trailing blanks
    on either side, prefixes are not equal, differences behind the first 8 bytes count, '' matches blanks"""
    import numpy as np
    vals = [b"BUILDING", b"BUILDING  ", b"BUILDIN", b"BUILDINGS", b"BUILDING X", b"", b" ", b"B", b"AUTOMOBILE", b"AUTOMOBILF",
            b"ABCDEFGHIJKL", b"ABCDEFGHIJKM", b"ABCDEFGH", b"ABCDEFGH    ", b"abcdefgh", b"MACHINERY", b"HOUSEHOLD", b"FURNITURE"]
    rng = np.random.default_rng(5)
    n = 70_001
    col = np.array([vals[i] for i in rng.integers(0, len(vals), n)], dtype="S13")
    ids = np.arange(n, dtype=np.int64)
    t = {"t": {"s": col, "i": ids}}
    h = engine.upload("t", t["t"])
    try:
        for const in (b"BUILDING", b"BUILDING ", b"ABCDEFGHIJKL", b"ABCDEFGH", b"", b"B", b"AUTOMOBILE", b"NOPE", b"ABCDEFGHIJKLMNOP"):
            for op in (16, 18):          # EQ_CHAR, NEQ_CHAR
                pool = const + b"\0"
                d = {"tables": [{"name": "t", "columns": ["s", "i"]}],
                     "pipelines": [{"source_kind": 1, "source_id": 0, "source_id2": 0, "sink_kind": 1, "size_hint": 0,
                                    "nodes": [[1, 0, 0, 0, 0], [1, 1, 0, 0, 0], [3, 0, 0, 0, 0], [op, 0, 2, 0, 0], [22, 3, 0, 0, 0]],
                                    "args": [], "keys": [], "vals": [[1, 2, 4, 0], [1, 1, 4, 0]]},
                                   {"source_kind": 2, "source_id": 0, "source_id2": 0, "sink_kind": 3, "size_hint": 0,
                                    "nodes": [[1, 0, 0, 0, 0], [1, 1, 0, 0, 0]], "args": [], "keys": [],
                                    "vals": [[0, 0, 4, 0], [1, 0, 4, 0]]}],
                     "order": [], "limit": -1, "strpool": pool.decode("latin1"), "result_names": ["n", "s"], "result_types": ["BIGINT"] * 2}
                res, _ = engine.execute(Plan(d), {"t": h})
                got = serialize_columns(res.columns, res.sql_types, res.sql_widths)
                want = serialize_columns(*run_plan(d, t))
                assert got == want, f"{const!r} op {op}: {got} != {want}"
    finally:
        h.free()


@pytest.mark.parametrize("limit", [0, 1, 7, 100000])
def test_limit_without_order_by_keeps_that_many_rows_of_the_result(limit, sf001, engine):
    """LIMIT without ORDER BY (materialize.h:135-140; Relation::applyLimit dbdata.h:407-425): WHICH rows
    survive is up to the scan order (per thread in the reference), but there are exactly min(limit, n) of
    them and each belongs to the unlimited result"""
    d = dict(load_plan_dict("sel_or"), order=[])          # the fixture's plan without its ORDER BY
    tabs = plan_tables(d, sf001)
    full, _ = _run(engine, d, tabs)
    d2 = dict(d, limit=limit)
    got, _ = _run(engine, d2, tabs)
    assert len(got) == min(limit, len(full))
    pool = {}
    for line in full:
        pool[line] = pool.get(line, 0) + 1
    for line in got:
        assert pool.get(line, 0) > 0, line
        pool[line] -= 1


def test_row_store_upload_matches_columns(sf001, engine):
    """rq_table_upload_rows (the bulk-insert hook) transposes reference DataBlocks on the GPU"""
    d = load_plan_dict("q1")
    cols = sf001["lineitem"]
    rows = tpch.to_rows("lineitem", cols)
    dt = rows.dtype
    names = d["tables"][0]["columns"]
    types, widths, offsets = [], [], []
    for n in names:
        kind, arg = next((k, a) for (c, k, a) in tpch.SCHEMAS["lineitem"] if c == n)
        cd = tpch.col_dtype(kind, arg)
        types.append({1: 1, 4: 2, 8: 3}[cd.itemsize] if cd.kind != "S" else 4)
        widths.append(cd.itemsize)
        offsets.append(dt.fields[n][1])
    raw = rows.tobytes()
    per_block = (2 << 20) // dt.itemsize * dt.itemsize     # DataBlock::Size = 2 MiB, whole tuples
    blocks = [raw[i:i + per_block] for i in range(0, len(raw), per_block)]
    t = engine.upload_rows("lineitem", names, types, widths, offsets, dt.itemsize, blocks)
    try:
        res, _ = engine.execute(Plan(d), {"lineitem": t})
    finally:
        t.free()
    got = serialize_columns(res.columns, res.sql_types, res.sql_widths)
    _, want = load_golden("q1")
    assert_same_relation(got, want, d, "q1 via row store")


def test_division_by_zero_is_reported(engine):
    d = {"tables": [{"name": "t", "columns": ["a", "b"]}],
         "pipelines": [{"source_kind": 1, "source_id": 0, "sink_kind": 3, "size_hint": 0,
                        "nodes": [[1, 0, 0, 0, 0], [1, 1, 0, 0, 0], [7, 0, 1, 0, 0]], "args": [], "keys": [],
                        "vals": [[2, 0, 4, 0]]}],
         "order": [], "limit": -1, "strpool": "", "result_names": ["q"], "result_types": ["BIGINT"]}
    from resql_b200 import EngineError
    t = engine.upload("t", {"a": np.arange(10, dtype=np.int64), "b": np.array([1] * 9 + [0], dtype=np.int64)})
    try:
        with pytest.raises(EngineError):
            engine.execute(Plan(d), {"t": t})
    finally:
        t.free()


def test_host_front_end_end_to_end(sf001, tmp_path):
    """The drop-in itself: the reference's parser/planner + our shim + the C ABI (prebuilt
    resql-b200) on the reference's row store, compared with the reference engine's output."""
    exe = os.path.join(ROOT, "resql_b200/host/resql-b200")
    if not os.path.exists(exe):
        pytest.skip("resql-b200 not built (needs the reference checkout at build time)")
    from golden.queries import QUERIES
    create = tmp_path / "create.sql"
    stm = []
    for name, schema in tpch.SCHEMAS.items():
        if name not in sf001:
            continue
        fields = []
        for c, k, a in schema:
            ty = {"int": "int", "date": "date", "bigint": "bigint"}.get(k) or (f"decimal(12,{a})" if k == "dec" else f"{k}({a})")
            fields.append(f"{c} {ty}")
        stm.append(f"create table {name} ( " + ", ".join(fields) + " )")
    create.write_text(";\n".join(stm) + ";\n")
    loads = [f"exec {create}"]
    for name, cols in sf001.items():
        p = tmp_path / f"{name}.bin"
        tpch.to_rows(name, cols).tofile(p)
        loads.append(f"binload {name} {p}")
    for q in ("q6", "q1", "q3", "q5", "q10", "q12", "q14", "sel_or", "agg_neg_avg", "micro_join_avg", "join_dups_agg", "nlj_cross_agg", "nlj_cross_filter"):
        out = tmp_path / f"{q}.out"
        sql = " ".join(QUERIES[q].split())
        r = subprocess.run([exe, "--quiet"] + loads + [f"out {out}", sql], capture_output=True, text=True, timeout=300)
        assert "#select" in r.stdout, r.stdout + r.stderr
        got = [l for l in out.read_text().split("\n")[1:] if l]
        _, want = load_golden(q)
        assert_same_relation(got, want, load_plan_dict(q), q + " via resql-b200")


def _join_plans():
    return [n for n in plan_names() if any(p["sink_kind"] == 2 for p in load_plan_dict(n)["pipelines"])]


@pytest.mark.parametrize("name", _join_plans())
def test_two_pass_probe_matches_reference_engine(name, sf001, engine):
    """selective probes run as scan -> Bloom test -> materialize, then a dense probe pass
    (engine_exec.inl split_at_probe); forced here for every join fixture regardless of size"""
    engine.set_option("split_min_rows", 0)
    engine.set_option("split_frac", 1e18)
    d = load_plan_dict(name)
    try:
        got, tm = _run(engine, d, plan_tables(d, sf001))
    finally:
        engine.set_option("split_min_rows", -1)
        engine.set_option("split_frac", -1)
    _, want = load_golden(name)
    assert_same_relation(got, want, d, name + " (two-pass)")
    n_scans = sum(1 for p in d["pipelines"] if p["source_kind"] == 1)
    assert tm.kernel_launches > n_scans


@pytest.mark.parametrize("limit", [1, 10, 100, 2048])
@pytest.mark.parametrize("name", ["sort_large", "sort_strings_large", "agg_many_groups"])
def test_order_by_limit_selects_top_k(name, limit, sf001, engine):
    """ORDER BY ... LIMIT k over more than 4096 rows takes the radix-select path (k-th smallest first
    key on the device, then a small sort of the candidates); the ORDER BY keys of these fixtures
    form a total order, so the first k rows are unique and must equal the oracle's"""
    d = dict(load_plan_dict(name))
    d["limit"] = limit
    tabs = plan_tables(d, sf001)
    got, _ = _run(engine, d, tabs)
    want = serialize_columns(*run_plan(d, tabs))
    assert len(got) == limit
    assert got == want


@pytest.mark.parametrize("name", ["q1", "q6", "q3", "q5", "q10", "sort_large", "agg_many_groups", "join_dups_rows", "nlj_cross_agg"])
def test_replayed_execution_is_identical_and_sync_free(name, sf001, engine):
    """The first clean execution records what the host read from the device; later executions of
    the same plan on the same tables predict those values and wait for the device exactly once, at
    the end (engine_exec.inl "host reads of device values"). Results must not change."""
    d = load_plan_dict(name)
    tabs = plan_tables(d, sf001)
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
    _, want = load_golden(name)
    for got, _ in runs:
        assert_same_relation(got, want, d, name + " (repeated)")
    assert runs[0][1].host_syncs >= 1
    assert runs[-1][1].host_syncs == 1, f"replay waited {runs[-1][1].host_syncs} times"
    assert runs[-1][1].kernel_launches > 0 and runs[-1][1].kernel_ms > 0      # graph launches still report device times


def test_replay_notices_changed_data_and_errors(engine):
    """Same table name, same row count, other contents: the predicted values are wrong, the replayed
    result is discarded and the plan runs the careful way - including error reporting."""
    from resql_b200 import EngineError
    d = {"tables": [{"name": "t", "columns": ["a", "b"]}],
         "pipelines": [{"source_kind": 1, "source_id": 0, "sink_kind": 1, "size_hint": 0,
                        "nodes": [[1, 0, 0, 0, 0], [1, 1, 0, 0, 0], [7, 0, 1, 0, 0]], "args": [],
                        "keys": [[1, 0, 4, 0]], "vals": [[2, 1, 4, 0], [0, 2, 4, 0]]}],
         "order": [[0, 1]], "limit": -1, "strpool": ""}
    n = 5000
    a = np.arange(n, dtype=np.int64) * 7
    variants = [np.full(n, 3, dtype=np.int64), (np.arange(n, dtype=np.int64) % 5) + 1, (np.arange(n, dtype=np.int64) % 900) + 1]
    for b in variants:
        t = engine.upload("t", {"a": a, "b": b})
        try:
            for _ in range(3):
                res, _ = engine.execute(Plan(d), {"t": t})
                got = serialize_columns(res.columns, res.sql_types, res.sql_widths)
                want = serialize_columns(*run_plan(d, {"t": {"a": a, "b": b}}))
                assert got == want
        finally:
            t.free()
    bz = variants[0].copy()
    bz[n // 2] = 0
    t = engine.upload("t", {"a": a, "b": bz})
    try:
        with pytest.raises(EngineError):
            engine.execute(Plan(d), {"t": t})
    finally:
        t.free()


def test_reference_suites_pass_through_the_gpu_shim():
    """The reference's OWN test suites (test/test_datatypes.h, test_expressions.h, test_operators.h;
    hand-built RelOperator trees checked by executeSelectAndCheckRelation, test_common.h:222) with
    executeSelectPlan routed to executeSelectPlanGpu: resql_b200/host/ref_tests_gpu.cpp, prebuilt
    in the container that has the reference checkout."""
    exe = os.path.join(ROOT, "resql_b200/host/resql-reftests-gpu")
    if not os.path.exists(exe):
        pytest.skip("resql-reftests-gpu not built (needs the reference checkout at build time)")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "ALL REFERENCE SUITES PASSED ON THE GPU PATH" in r.stdout
    assert r.stdout.count(" OK") >= 40
