"""Late materialization without a GPU: rq_debug_lower with IMPL_LATE prints the record layout of a
materialize pipeline (references, computed outputs, deferred columns and their origin) and then
the record pipeline lowered as IMPL_EMIT. Wide synthetic shapes that the early form refuses must
lower, staging only the columns the program reads."""
import pytest

from resql_b200 import EngineError, Plan
from resql_b200 import native as N
from resql_b200.plan import OP

IMPL_EMIT, IMPL_LATE = 4, 7
I8, I32, I64, STR = N.RQ_I8, N.RQ_I32, N.RQ_I64, N.RQ_STR


def wide_select(types, filter_lt=None, computed=False):
    """select * [, c1 + c2] from w [where c0 < k]"""
    n = len(types)
    nodes = [[OP["COL"], i, 0, 0, 0] for i in range(n)]
    if filter_lt is not None:
        nodes.append([OP["CONST"], 0, 0, 0, filter_lt])
        nodes.append([OP["LT"], 0, n, 0, 0])
        nodes.append([OP["FILTER"], n + 1, 0, 0, 0])
    vals = [[i, 0, 4, 0] for i in range(n)]
    if computed:
        nodes.append([OP["ADD"], 1, 2, 0, 0])
        vals.append([len(nodes) - 1, 0, 4, 0])
    p = {"source_kind": 1, "source_id": 0, "sink_kind": 3, "size_hint": 0, "args": [], "nodes": nodes,
         "keys": [], "vals": vals}
    return {"tables": [{"name": "w", "columns": [f"c{i}" for i in range(n)]}], "pipelines": [p],
            "order": [], "limit": -1, "strpool": ""}


def types_of(n):
    """columns 0, 1 and 2 int64 (filter / computed operands), then a mix: 17 columns hold 17 fixed-width
    ones, 40 and 64 more than 8 strings"""
    if n == 17:
        return [(I64, 8)] * 3 + [((I32, 4), (I8, 1))[i % 2] for i in range(n - 3)]
    mix = [(I32, 4), (I8, 1), (STR, 6), (I64, 8), (STR, 13)]
    return [(I64, 8)] * 3 + [mix[i % len(mix)] for i in range(n - 3)]


def lower(d, impl, tw):
    return N.debug_lower(Plan(d), 0, impl, [t for t, _ in tw], [w for _, w in tw])


def parse(out):
    lines = out.splitlines()
    refs = [l.split()[2:] for l in lines if l.startswith("ref ")]
    outs = [l.split() for l in lines if l.startswith(("computed ", "deferred "))]
    head = next(l.split() for l in lines if l.startswith("cols "))
    return refs, outs, dict(zip(head[0::2], map(int, head[1::2]))), lines


@pytest.mark.parametrize("n", [12, 17, 40, 64])
@pytest.mark.parametrize("computed", [False, True])
@pytest.mark.parametrize("filt", [None, 5])
def test_wide_select_star_lowers_late(n, computed, filt):
    tw = types_of(n)
    d = wide_select(tw, filt, computed)
    n_str = sum(t == STR for t, _ in tw)
    if n > 24 or n - n_str > 16 or n_str > 8:      # beyond the early form
        with pytest.raises(EngineError) as e:
            lower(d, IMPL_EMIT, tw)
        assert e.value.code == 3
    refs, outs, head, lines = parse(lower(d, IMPL_LATE, tw))
    assert refs == [["row"]]
    assert [o[:3] for o in outs[:n]] == [["deferred", str(k), "col"] for k in range(n)]
    assert [int(o[3]) for o in outs[:n]] == list(range(n))
    if computed:
        assert outs[n] == ["computed", str(n), "rec", "1"]
    # staged: only what the program and the computed output read; no string operands
    want_cols = {0} if filt is not None else set()
    if computed:
        want_cols |= {1, 2}
    assert head["cols"] == len(want_cols) and head["strcols"] == 0
    staged = {int(l.split()[3]) for l in lines if l.startswith("col ")}
    assert staged == want_cols
    # the record: the row index (slot 0, written by the kernel), then the computed output
    assert head["nout"] == 1 + (1 if computed else 0)
    assert any(l == "late_row 1 0" for l in lines)


def test_narrow_select_has_the_same_record_shape():
    tw = types_of(5)
    refs, outs, head, _ = parse(lower(wide_select(tw, 3, True), IMPL_LATE, tw))
    assert refs == [["row"]] and len(outs) == 6 and head["nout"] == 2


def test_pipeline_without_deferrable_output_has_no_late_form():
    tw = types_of(4)
    d = wide_select(tw, None, True)
    d["pipelines"][0]["vals"] = d["pipelines"][0]["vals"][-1:]
    with pytest.raises(EngineError) as e:
        lower(d, IMPL_LATE, tw)
    assert e.value.code == 3
