"""Generates tests/golden/loader_sf002.json: what a `select <all columns>` returns after the `.tbl` files of
tests/test_gpu_loader.py (generated tables with edited edge cases) are bulk-inserted, summarized per table by
test_gpu_loader.golden_summary. The rows come from the reference engine (oracle/_ref/resql-oracle, built by
oracle/ref_build/build_ref.sh) when it is built, otherwise from rq_table_load_tbl of a build whose loader
test passed against the reference engine; "source" records which. Needs a GPU in the second case.

    python tests/golden/make_loader_golden.py
"""
import json
import os
import subprocess
import sys
import tempfile
from pathlib import Path

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import test_gpu_loader as L  # noqa: E402

ORACLE = os.path.join(ROOT, "oracle/_ref/resql-oracle")


def main():
    data = L.edited_tables()
    out = {}
    engine = None
    with tempfile.TemporaryDirectory() as tmp:
        for table in ("customer", "orders", "lineitem"):
            p = Path(tmp) / f"{table}.tbl"
            L.write_edited_tbl(table, data, p)
            if os.path.exists(ORACLE):
                source = "reference engine: bulk insert, then select <all columns>"
                create, res = Path(tmp) / "create.sql", Path(tmp) / f"{table}.out"
                create.write_text(L._create_sql([table]))
                cols = ", ".join(s[0] for s in L.sql_schema(table))
                subprocess.run([ORACLE, "--quiet", f"exec {create}", f'bulk insert {table} from "{p}" with ( fieldterminator="|" )',
                                f"out {res}", f"select {cols} from {table}"], check=True, capture_output=True, timeout=600)
                lines = [l for l in res.read_text(encoding="latin1").split("\n")[1:] if l]
            else:
                from resql_b200 import Engine
                source = "rq_table_load_tbl of a build that matched the reference engine's bulk insert"
                engine = engine or Engine(0)
                lines = L.load_and_select_all(engine, table, p)
            out[table] = L.golden_summary(table, data, lines)
    if engine is not None:
        engine.shutdown()
    with open(os.path.join(ROOT, "tests/golden/loader_sf002.json"), "w") as f:
        json.dump({"source": source, **out}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
