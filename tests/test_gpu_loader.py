"""rq_table_load_tbl: the parallel `.tbl` text loader (csrc/tbl_loader.inl; replaces the row-store fill of
executeBulkInsert, execute.h:332-388). The table it builds must hold exactly what the reference's own
`bulk insert` puts into its row store: checked through `select <all columns>` against the reference
engine on the same files (stored under tests/golden/loader_sf002.json), and against the columns the
files were written from."""
import hashlib
import json
import os
import subprocess

import pytest

from common import GOLDEN, ROOT, assert_same_relation, load_plan_dict, serialize_columns
from resql_b200 import Plan, tpch

pytestmark = pytest.mark.gpu

SQL_OF = {"int": 3, "date": 7, "bigint": 4, "dec": 5}


def sql_schema(table):
    out = []
    for c, k, a in tpch.SCHEMAS[table]:
        if k in SQL_OF:
            out.append((c, SQL_OF[k], 0, 12 * 256 + a if k == "dec" else 0))
        else:
            out.append((c, 1 if k == "char" else 0, a, a))
    return out          # (column, RQ_SQL type, n of CHAR/VARCHAR, rq_value width)


def select_all(table):
    sch = sql_schema(table)
    return {"tables": [{"name": table, "columns": [s[0] for s in sch]}],
            "pipelines": [{"source_kind": 1, "source_id": 0, "source_id2": 0, "sink_kind": 3, "size_hint": 0,
                           "nodes": [[1, i, 0, 0, 0] for i in range(len(sch))], "args": [], "keys": [],
                           "vals": [[i, 0, s[1], s[3]] for i, s in enumerate(sch)]}],
            "order": [], "limit": -1, "strpool": "", "result_names": [s[0] for s in sch], "result_types": [""] * len(sch)}


@pytest.fixture(scope="module")
def engine():
    from resql_b200 import Engine
    eng = Engine(0)
    yield eng
    eng.shutdown()


def _create_sql(tables):
    stm = []
    for name in tables:
        fields = []
        for c, k, a in tpch.SCHEMAS[name]:
            ty = {"int": "int", "date": "date", "bigint": "bigint"}.get(k) or (f"decimal(12,{a})" if k == "dec" else f"{k}({a})")
            fields.append(f"{c} {ty}")
        stm.append(f"create table {name} ( " + ", ".join(fields) + " )")
    return ";\n".join(stm) + ";\n"


def edited_tables():
    """the tables of the bulk-insert test, with edge cases the generator does not produce: negative and
    point-free decimals, yyyy/mm/dd dates, strings longer than the column, a last line without a line end"""
    data = tpch.generate(0.02, seed=77, tables=("lineitem", "orders", "customer"))
    cust = {c: v.copy() for c, v in data["customer"].items()}
    cust["c_acctbal"][:4] = [-99999, -5, 0, 123456789]
    data["customer"] = cust
    return data


def write_edited_tbl(table, data, p):
    tpch.write_tbl(table, data[table], p)
    text = p.read_text(encoding="latin1")
    if table == "orders":
        lines = text.split("\n")
        lines[0] = lines[0].replace("-", "/", 2)                   # date written as yyyy/mm/dd
        text = "\n".join(lines)
    if table == "customer":
        first = text.split("\n")[0].split("|")
        first[1] = first[1] + "x" * 40                              # longer than VARCHAR(25): cut by the loader
        first[5] = "42"                                              # decimal literal without a point
        text = "|".join(first) + "\n" + text.split("\n", 1)[1]
        text = text.rstrip("\n")                                     # no line end behind the last row
    p.write_text(text, encoding="latin1")


def load_and_select_all(engine, table, p):
    sch = sql_schema(table)
    h = engine.load_tbl(table, p, [(s[0], s[1], s[2]) for s in sch])
    try:
        res, _ = engine.execute(Plan(select_all(table)), {table: h})
    finally:
        h.free()
    return serialize_columns(res.columns, res.sql_types, res.sql_widths)


def golden_summary(table, data, lines):
    """what tests/golden/loader_sf002.json stores of a `select <all columns>`: the row count, a digest of
    the sorted rows and, readable, the rows of the edited keys"""
    keys = {str(int(k)) for k in data[table][tpch.SCHEMAS[table][0][0]][:4]}
    rows = sorted(lines)
    return {"rows": len(rows), "sha256": hashlib.sha256("\n".join(rows).encode("latin1")).hexdigest(),
            "edited_rows": [l for l in rows if l.split("|")[0] in keys]}


def test_loaded_tables_equal_the_reference_bulk_insert(engine, tmp_path):
    data = edited_tables()
    with open(os.path.join(GOLDEN, "loader_sf002.json")) as f:
        golden = json.load(f)
    ref = os.path.join(ROOT, "oracle/_ref/resql-oracle")
    for table in ("customer", "orders", "lineitem"):
        p = tmp_path / f"{table}.tbl"
        write_edited_tbl(table, data, p)
        sch = sql_schema(table)
        got = load_and_select_all(engine, table, p)
        assert len(got) == len(data[table][sch[0][0]])
        # the reference's `bulk insert` of the same file, stored: the edited rows verbatim, all rows as a digest
        summary = golden_summary(table, data, got)
        assert summary["edited_rows"] == golden[table]["edited_rows"], table
        assert summary == golden[table], f"{table}: loaded rows differ from the reference's bulk insert"
        if os.path.exists(ref):
            out = tmp_path / f"{table}.out"
            create = tmp_path / "create.sql"
            create.write_text(_create_sql([table]))
            cols = ", ".join(s[0] for s in sch)
            r = subprocess.run([ref, "--quiet", f"exec {create}", f'bulk insert {table} from "{p}" with ( fieldterminator="|" )',
                                f"out {out}", f"select {cols} from {table}"], capture_output=True, text=True, timeout=600)
            want = [l for l in out.read_text(encoding="latin1").split("\n")[1:] if l]
            # (a select without ORDER BY returns the rows in any order: compare as multisets, test_common.h:125-190)
            assert sorted(got) == sorted(want), f"{table}: first difference {[(a, b) for a, b in zip(sorted(got), sorted(want)) if a != b][:2]}"
        if table == "lineitem":      # untouched file: the loaded table is the generated one
            want = serialize_columns([data[table][s[0]] for s in sch], [s[1] for s in sch], [s[3] for s in sch])
            assert sorted(got) == sorted(want)


def test_reference_query_suite_on_loaded_tbl_files(engine, tmp_path):
    """test/test_queries.h:5-110 on tables built by the loader: the SF0.01 `.tbl` files the reference ships
    plus the lineitem table regenerated by resql_b200/dbgen.py, loaded with rq_table_load_tbl; the seven
    statements must give the reference's golden results (test/reference/q*.tbl, copies under
    tests/golden/dbgen_sf001)."""
    import gzip
    from resql_b200 import dbgen
    D = os.path.join(GOLDEN, "dbgen_sf001")
    handles = {}
    try:
        for name in ("lineitem", "orders", "customer", "supplier", "part", "nation", "region"):
            p = tmp_path / f"{name}.tbl"
            if name == "lineitem":
                tpch.write_tbl("lineitem", dbgen.generate_orders_lineitem(0.01)[1], p)
            else:
                with gzip.open(os.path.join(D, name + ".tbl.gz"), "rb") as f:
                    p.write_bytes(f.read())
            handles[name] = engine.load_tbl(name, p, [(s[0], s[1], s[2]) for s in sql_schema(name)])
        for q in ("q1", "q3", "q5", "q6", "q10", "q12", "q19"):
            d = load_plan_dict(q)
            res, _ = engine.execute(Plan(d), {t["name"]: handles[t["name"]] for t in d["tables"]})
            got = serialize_columns(res.columns, res.sql_types, res.sql_widths)
            with open(os.path.join(D, q + ".tbl")) as f:
                want = [l for l in f.read().split("\n") if l]
            assert_same_relation(got, want, d, f"{q}: loaded dbgen SF0.01 files vs test/reference/{q}.tbl")
    finally:
        for h in handles.values():
            h.free()


def test_malformed_lines_are_reported_like_the_reference(engine, tmp_path):
    from resql_b200 import EngineError
    sch = [("a", 3, 0), ("b", 5, 0)]
    for text, msg in (("1|2.5|\n2|\n3|1.0|\n", "missing attributes"), ("1|2.5|\n2|3.5|4|\n", "extra attributes"), ("1|2.5|\n\n", "missing attributes")):
        p = tmp_path / "bad.tbl"
        p.write_text(text)
        with pytest.raises(EngineError) as e:
            engine.load_tbl("t", p, sch)
        assert msg in str(e.value)
    with pytest.raises(EngineError):
        engine.load_tbl("t", tmp_path / "absent.tbl", sch)
