"""ORDER BY ... LIMIT plans over chosen key columns, an exact reference of what they return and a
tie-aware comparison, for test_order_plans.py and test_gpu_order_by.py. A plan scans table t (an
optional selection `col op const`) into one of three final relations: a materialize of chosen
columns; a GROUP BY aggregation followed by a projection of its keys and aggregates (the relation
comes out of a hash table); or an equi-join of t with a build table b, materialized. ORDER BY and
LIMIT then apply to that relation.

The reference restates the sort order of sort_kernels.cuh and plan_oracle.finish in plain numpy:
integers, DATE and DECIMAL compare as signed int64; CHAR(1) and BOOL as zero-extended bytes; CHAR(n>1)
and VARCHAR as unsigned bytes up to the NUL (strcmp, trailing blanks count); DESC per key. Its sort
is stable, but the engine's order inside ties is not specified, so results are compared with
assert_ordered_equal: the same sequence of ORDER BY key tuples, the same multiset of rows inside
every run of equal key tuples, and, where the LIMIT cuts a run, a sub-multiset of the reference's
whole run. Test infrastructure only."""
import numpy as np

from inlist_plans import Pipe, new_plan, SINK_AGG, SINK_BUILD, SINK_MAT
from plan_fuzz import (SQL_VARCHAR, SQL_CHAR, SQL_BOOL, SQL_INT, SQL_BIGINT, SQL_DECIMAL, SQL_DATE, AGG_SUM,
                       AGG_COUNT, AGG_MIN, AGG_MAX)

I64_MIN, I64_MAX = -2 ** 63, 2 ** 63 - 1
I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1
SRC_PIPE = 2
KEEP = {"LT": np.less, "LE": np.less_equal, "GT": np.greater, "GE": np.greater_equal, "EQ": np.equal}


class OrderCase:
    """t: {column: numpy array} (int64, int32, uint8 or S<w+1>); sql: {column: (sql type, width)} for
    columns whose type is not the default of their dtype (BIGINT, INT, CHAR(1), CHAR(w));
    out: the materialized columns; sel: (column, op, const) or None;
    group: ([key columns], [(AGG kind, column or None)]) - the projection after it outputs the
    columns of the aggregation in the order `out` names them by index;
    join: (b, [probe key, build key], [build payloads]) - b a table like t with unique keys;
    order: [(output column index, ascending)]; limit: -1 or k;
    path: the ORDER BY path the engine must take: "none" (nothing to sort), "bitonic", "radix",
    "topk" or "topk->radix"; passes: the radix digit passes the trace must report (None: any)."""

    def __init__(self, name, t, out, order, limit=-1, sql=None, sel=None, group=None, join=None, path=None,
                 passes=None):
        self.name, self.t, self.out, self.order, self.limit = name, t, list(out), [tuple(o) for o in order], limit
        self.sql_over, self.sel, self.group, self.join = dict(sql or {}), sel, group, join
        self.path, self.passes = path, passes

    @property
    def n(self):
        return len(next(iter(self.t.values())))

    def sql(self, col, table=None):
        a = (table if table is not None else self.t)[col]
        if col in self.sql_over:
            return self.sql_over[col]
        if a.dtype.kind == "S":
            return SQL_CHAR, a.dtype.itemsize - 1
        return {np.dtype(np.int64): (SQL_BIGINT, 0), np.dtype(np.int32): (SQL_INT, 0),
                np.dtype(np.uint8): (SQL_CHAR, 1)}[a.dtype]

    def tables(self):
        return {"t": self.t, **({"b": self.join[0]} if self.join else {})}


def is_str(sql):
    t, w = sql
    return t == SQL_VARCHAR or (t == SQL_CHAR and w > 1)


# ---- plans ---------------------------------------------------------------------------------------------
def _agg_sql(kind, sql):
    return (SQL_BIGINT, 0) if kind in (AGG_SUM, AGG_COUNT) else sql


def result_sql(c):
    """(sql type, width) of every column of the final relation"""
    if c.group:
        keys, aggs = c.group
        cols = [c.sql(k) for k in keys] + [_agg_sql(kind, c.sql(v) if v else None) for kind, v in aggs]
        return [cols[i] for i in c.out]
    if c.join:
        b, _, pay = c.join
        return [c.sql(o) for o in c.out] + [c.sql(p, b) for p in pay]
    return [c.sql(o) for o in c.out]


def order_plan(c, tag=0):
    """the plan of case c. tag: a dead constant in the scan of t, so that plans of cases that share
    their shape do not share the engine's memos of earlier executions"""
    tabs = {"t": list(c.t)}
    if c.join:
        tabs["b"] = list(c.join[0])
    d, pool = new_plan(tabs)
    if c.join:
        b, (pk, bk), pay = c.join
        bp = Pipe(d, "b", list(b), pool)
        bp.done(SINK_BUILD, [[bp.col(v), 0, *c.sql(v, b)] for v in pay], [[bp.col(bk), 0, *c.sql(bk, b)]])
    p = Pipe(d, "t", list(c.t), pool)
    p.const(9_000_000 + tag)
    if c.sel:
        col, op, k = c.sel
        p.filter(p.n(op, p.col(col), p.const(k)))
    if c.group:
        keys, aggs = c.group
        kv = [[p.col(k), 0, *c.sql(k)] for k in keys]
        vv = [[p.col(v) if v else p.const(1), kind, *_agg_sql(kind, c.sql(v) if v else None)] for kind, v in aggs]
        p.done(SINK_AGG, vv, kv)
        names = [f"g{i}" for i in range(len(kv) + len(vv))]
        sql = [x[2:] for x in kv + vv]
        q = Pipe(d, None, names, pool)
        q.done(SINK_MAT, [[q.col(names[i]), 0, *sql[i]] for i in c.out], source_kind=SRC_PIPE,
               source_id=len(d["pipelines"]) - 1)
    elif c.join:
        b, (pk, bk), pay = c.join
        p.args = [p.col(pk)]
        pr = p.n("PROBE", 0, 0, 1, 1)
        pays = [p.n("PAYLOAD", pr, j) for j in range(len(pay))]
        p.done(SINK_MAT, [[p.col(o), 0, *c.sql(o)] for o in c.out] + [[x, 0, *c.sql(v, b)] for x, v in zip(pays, pay)])
    else:
        p.done(SINK_MAT, [[p.col(o), 0, *c.sql(o)] for o in c.out])
    d["order"] = [[int(i), int(bool(asc))] for i, asc in c.order]
    d["limit"] = int(c.limit)
    return d


# ---- the reference ----------------------------------------------------------------------------------------
def _strings(a):
    return np.array([bytes(x).split(b"\0")[0] for x in a], dtype=object)


def _values(a):
    return _strings(a) if a.dtype.kind == "S" else a.astype(np.int64)


def final_relation(c):
    """the relation ORDER BY applies to, unordered: a list of columns (int64 arrays, object arrays of
    bytes), integers as the sink stores them (CHAR(1) / BOOL zero-extended)"""
    rows = np.arange(c.n)
    if c.sel:
        col, op, k = c.sel
        rows = rows[KEEP[op](c.t[col].astype(np.int64), k)]
    if c.join:
        b, (pk, bk), pay = c.join
        where = {int(x): i for i, x in enumerate(b[bk].astype(np.int64))}
        assert len(where) == len(b[bk]), "build keys must be unique"
        hit = [(r, where[int(x)]) for r, x in zip(rows, c.t[pk][rows].astype(np.int64)) if int(x) in where]
        pr = np.array([h[0] for h in hit], np.int64)
        br = np.array([h[1] for h in hit], np.int64)
        return [_values(c.t[o][pr]) for o in c.out] + [_values(b[v][br]) for v in pay]
    if not c.group:
        return [_values(c.t[o][rows]) for o in c.out]
    keys, aggs = c.group
    kv = [_values(c.t[k][rows]) for k in keys]
    codes = [np.unique(v, return_inverse=True)[1].reshape(-1) for v in kv]
    if len(rows) == 0:
        return [np.zeros(0, object if kv[i].dtype == object else np.int64) if i < len(keys) else np.zeros(0, np.int64)
                for i in c.out]
    _, first, gid = np.unique(np.stack(codes, axis=1), axis=0, return_index=True, return_inverse=True)
    gid = gid.reshape(-1)
    ng = len(first)
    cols = [v[first] for v in kv]
    for kind, v in aggs:
        if kind == AGG_COUNT:
            cols.append(np.bincount(gid, minlength=ng).astype(np.int64))
            continue
        x = c.t[v][rows].astype(np.int64)
        if kind == AGG_SUM:
            acc = np.zeros(ng, np.uint64)
            np.add.at(acc, gid, x.view(np.uint64))
            cols.append(acc.view(np.int64))
        else:
            acc = np.full(ng, I64_MAX if kind == AGG_MIN else I64_MIN, np.int64)
            (np.minimum if kind == AGG_MIN else np.maximum).at(acc, gid, x)
            cols.append(acc)
    return [cols[i] for i in c.out]


def sort_ranks(col):
    """int64 ranks that order like the column under strcmp / signed int64 compare"""
    return np.unique(col, return_inverse=True)[1].reshape(-1).astype(np.int64)


def reference(c):
    """the final relation of case c in ORDER BY order (stable inside ties), before the LIMIT"""
    cols = final_relation(c)
    n = len(cols[0]) if cols else 0
    if n == 0 or not c.order:
        return cols
    keys = [sort_ranks(cols[i]) * (1 if asc else -1) for i, asc in c.order]
    idx = np.lexsort(keys[::-1])
    return [x[idx] for x in cols]


def canonical(cols, sql):
    """result columns -> int64 arrays and object arrays of bytes (up to the NUL)"""
    return [(_strings(a) if np.asarray(a).dtype.kind == "S" else np.asarray(a)) if is_str(s)
            else np.asarray(a).astype(np.int64) for a, s in zip(cols, sql)]


def _codes(got, want):
    """both sides as int64 matrices, string columns replaced by their rank among the strings of both"""
    ng = len(got[0]) if got else 0
    g, w = [], []
    for x, y in zip(got, want):
        if x.dtype == object or y.dtype == object:
            r = sort_ranks(np.concatenate([np.asarray(x, object), np.asarray(y, object)]))
            x, y = r[:ng], r[ng:]
        g.append(np.asarray(x, np.int64))
        w.append(np.asarray(y, np.int64))
    return np.stack(g, axis=1), np.stack(w, axis=1)


def _sorted_rows(m):
    return m[np.lexsort(m.T[::-1])] if len(m) else m


def assert_ordered_equal(got, want_sorted, sql, order, limit, what=""):
    """got: the engine's result columns; want_sorted: reference(c) (the whole relation, ordered).
    Fails unless got is one of the results ORDER BY ... LIMIT allows: the sequence of ORDER BY key
    tuples equals the reference's first rows', each maximal run of equal key tuples holds the same
    multiset of rows, and the run the LIMIT cuts holds a sub-multiset of the reference's whole run."""
    got, want = canonical(got, sql), canonical(want_sorted, sql)
    n = len(want[0]) if want else 0
    k = n if limit < 0 else min(limit, n)
    ng = len(got[0]) if got else 0
    assert ng == k, f"{what}: {ng} rows, the reference keeps {k} of {n}"
    if k == 0:
        return
    g, w = _codes(got, want)
    kc = [i for i, _ in order]
    bad = np.flatnonzero((g[:, kc] != w[:k, kc]).any(axis=1)) if kc else []
    assert len(bad) == 0, (f"{what}: the ORDER BY key sequence differs first at row {bad[0]} of {k}: "
                           f"{g[bad[0], kc].tolist()} vs {w[bad[0], kc].tolist()}")
    # runs of equal key tuples over the reference's whole relation; `cut` starts the run the LIMIT cuts
    if kc:
        change = np.flatnonzero((w[1:, kc] != w[:-1, kc]).any(axis=1)) + 1
        starts = np.concatenate([[0], change])
    else:
        starts = np.zeros(1, np.int64)
    run = np.searchsorted(starts, np.arange(n), "right") - 1
    ends = np.concatenate([starts[1:], [n]])
    cut = starts[run[k - 1]] if ends[run[k - 1]] > k else k
    full_g = _sorted_rows(np.column_stack([run[:cut], g[:cut]]))
    full_w = _sorted_rows(np.column_stack([run[:cut], w[:cut]]))
    bad = np.flatnonzero((full_g != full_w).any(axis=1))
    assert len(bad) == 0, (f"{what}: the rows inside a run of equal ORDER BY keys differ ({len(bad)} of {cut}), "
                           f"first {full_g[bad[0], 1:].tolist()} vs {full_w[bad[0], 1:].tolist()}")
    if cut < k:
        e = ends[run[k - 1]]
        rows, inv = np.unique(np.concatenate([g[cut:k], w[cut:e]]), axis=0, return_inverse=True)
        inv = inv.reshape(-1)
        have = np.bincount(inv[:k - cut], minlength=len(rows))
        may = np.bincount(inv[k - cut:], minlength=len(rows))
        over = np.flatnonzero(have > may)
        assert len(over) == 0, (f"{what}: the LIMIT cuts a run of {e - cut} equal keys after {k - cut} rows, and "
                                f"row {rows[over[0]].tolist()} is not one of the run's (or too often)")


__all__ = ["OrderCase", "order_plan", "result_sql", "final_relation", "reference", "assert_ordered_equal",
           "I64_MIN", "I64_MAX", "I32_MIN", "I32_MAX", "SQL_VARCHAR", "SQL_CHAR", "SQL_BOOL", "SQL_INT", "SQL_BIGINT",
           "SQL_DECIMAL", "SQL_DATE", "AGG_SUM", "AGG_COUNT", "AGG_MIN", "AGG_MAX"]
