"""Equi-join plans over chosen key columns, and an exact numpy reference of what they return, for
test_gpu_join_keys.py. A plan is one BUILD pipeline over table b and one probe pipeline over table p
that either materializes the joined rows or aggregates over them (COUNT(*), SUM of a build payload,
SUM of a probe value; ungrouped or grouped by the probe key). The reference joins by sorting the
build keys and searching the probe keys in them; CHAR keys compare after their trailing blanks are
stripped, VARCHAR keys exactly, integer keys as int64 whatever their width. Sums wrap around 2^64.
Test infrastructure only."""
import numpy as np

from inlist_plans import Pipe, new_plan, SINK_AGG, SINK_BUILD, SINK_MAT
from plan_fuzz import SQL_VARCHAR, SQL_CHAR, SQL_INT, SQL_BIGINT, AGG_SUM, AGG_COUNT

I64_MIN, I64_MAX = -2 ** 63, 2 ** 63 - 1
HALF_MIN, HALF_MAX = -2 ** 62, 2 ** 62 - 1        # INT64_MIN / 2 and INT64_MAX / 2 in C
FIB = 0x9E3779B97F4A7C15                           # the multiplier of hash_int (hash_kernels.cuh)
FIB_INV = pow(FIB, -1, 2 ** 64)


def home_slot(key, capacity):
    """the home slot of an integer key in a hash-form join table of `capacity` (a power of two)
    slots: the top log2(capacity) bits of key * FIB mod 2^64"""
    lg = capacity.bit_length() - 1
    return ((key % 2 ** 64) * FIB % 2 ** 64) >> (64 - lg)


def key_of_hash(h):
    """the int64 key whose hash is h (h * FIB^-1 mod 2^64)"""
    k = h * FIB_INV % 2 ** 64
    return k - 2 ** 64 if k >= 2 ** 63 else k


class JoinCase:
    """build, probe: {column: numpy array}; bkeys / pkeys: the join key columns of each side, in the
    same order; pay: build columns carried as payloads (a join key column among them is the key
    value itself); out: probe columns of a materialized row (agg None), or agg "all" / "by_key"
    (COUNT(*), SUM(pay[0]), SUM(probe column `pval`)); filters: [(build column, op, const,
    const_on_left)]; varchar: string keys and payloads are VARCHAR rather than CHAR.
    path: the build form the engine takes with direct-address joins on: "direct", "dup" (direct,
    then the hash form after a duplicate key), "hash" or "grow" (hash form, regrown); expand: a probe
    tuple meets more than one entry."""

    def __init__(self, name, build, probe, bkeys, pkeys, pay, out=(), agg=None, pval=None, single=0, filters=(),
                 size_hint=0, varchar=False, path="hash", expand=False):
        self.name, self.build, self.probe = name, build, probe
        self.bkeys, self.pkeys, self.pay, self.out = list(bkeys), list(pkeys), list(pay), list(out)
        self.agg, self.pval, self.single, self.filters = agg, pval, single, list(filters)
        self.size_hint, self.varchar, self.path, self.expand = size_hint, varchar, path, expand

    def sql(self, col):
        """(sql type, width) of a column of either table"""
        a = self.build[col] if col in self.build else self.probe[col]
        if a.dtype.kind == "S":
            return (SQL_VARCHAR if self.varchar else SQL_CHAR), a.dtype.itemsize - 1
        return {np.dtype(np.int64): (SQL_BIGINT, 0), np.dtype(np.int32): (SQL_INT, 0), np.dtype(np.uint8): (SQL_CHAR, 1)}[a.dtype]

    def is_str(self, col):
        t, w = self.sql(col)
        return t == SQL_VARCHAR or (t == SQL_CHAR and w > 1)


# ---- plans ---------------------------------------------------------------------------------------------
def join_plan(c, tag=0):
    """the plan of case c. tag: a dead constant in the build pipeline and an always true selection
    `pid > -1 - tag` behind the probe (where the second pass of a split probe keeps it), so that the
    engine's memos of earlier executions (build form, table capacity, expansion) do not apply"""
    d, pool = new_plan({"b": list(c.build), "p": list(c.probe)})
    b = Pipe(d, "b", list(c.build), pool)
    node = {}

    def col(name):
        if name not in node:
            node[name] = b.col(name)
        return node[name]
    for k in c.bkeys:
        col(k)
    for f, op, k, left in c.filters:
        x, y = col(f), b.const(k)
        b.filter(b.n(op, y, x) if left else b.n(op, x, y))
    keys = [[col(k), 0, *c.sql(k)] for k in c.bkeys]
    vals = [[col(v), 0, *c.sql(v)] for v in c.pay]
    b.const(7_000_000 + tag)
    b.done(SINK_BUILD, vals, keys)
    d["pipelines"][-1]["size_hint"] = c.size_hint

    p = Pipe(d, "p", list(c.probe), pool)
    pk = [p.col(k) for k in c.pkeys]
    p.args = list(pk)
    pr = p.n("PROBE", 0, 0, len(pk), c.single)
    pay = [p.n("PAYLOAD", pr, j) for j in range(len(c.pay))]
    p.filter(p.n("GT", p.col("pid"), p.const(-1 - tag)))
    if c.agg is None:
        vals = [[p.col(o), 0, *c.sql(o)] for o in c.out] + [[pay[j], 0, *c.sql(v)] for j, v in enumerate(c.pay)]
        keys = []
        sink = SINK_MAT
    else:
        vals = [[0, AGG_COUNT, SQL_BIGINT, 0], [pay[0], AGG_SUM, SQL_BIGINT, 0], [p.col(c.pval), AGG_SUM, SQL_BIGINT, 0]]
        keys = [[p.col(c.pkeys[0]), 0, SQL_BIGINT, 0]] if c.agg == "by_key" else []
        sink = SINK_AGG
    p.done(sink, vals, keys)
    return d


def result_sql(c):
    """(sql type, width) of every result column"""
    if c.agg is None:
        return [c.sql(o) for o in c.out] + [c.sql(v) for v in c.pay]
    return ([(SQL_BIGINT, 0)] if c.agg == "by_key" else []) + [(SQL_BIGINT, 0)] * 3


# ---- the reference ----------------------------------------------------------------------------------------
def _strings(a):
    return np.array([bytes(x).split(b"\0")[0] for x in a], dtype=object)


def _key_values(c, side, col):
    a = (c.build if side == "b" else c.probe)[col]
    if a.dtype.kind != "S":
        return a.astype(np.int64)
    s = _strings(a)
    if not c.varchar:                  # compareChar: trailing blanks do not count
        s = np.array([x.rstrip(b" ") for x in s], dtype=object)
    return s


def key_codes(c):
    """one int64 code per build row and per probe row, equal exactly where their join keys are"""
    nb = len(next(iter(c.build.values())))
    code = None
    for bk, pk in zip(c.bkeys, c.pkeys):
        both = np.concatenate([_key_values(c, "b", bk), _key_values(c, "p", pk)])
        inv = np.unique(both, return_inverse=True)[1].reshape(-1).astype(np.int64)
        code = inv if code is None else np.unique(np.stack([code, inv], axis=1), axis=0, return_inverse=True)[1].reshape(-1)
    return code[:nb], code[nb:]


def build_passes(c):
    """the build rows that pass the build filters"""
    nb = len(next(iter(c.build.values())))
    keep = np.ones(nb, bool)
    for f, op, k, left in c.filters:
        x = c.build[f].astype(np.int64)
        op = {"LT": "GT", "LE": "GE", "GT": "LT", "GE": "LE", "EQ": "EQ"}[op] if left else op
        keep &= {"LT": x < k, "LE": x <= k, "GT": x > k, "GE": x >= k, "EQ": x == k}[op]
    return np.flatnonzero(keep)


def _column(c, side, col, idx):
    a = (c.build if side == "b" else c.probe)[col][idx]
    return _strings(a) if a.dtype.kind == "S" else a.astype(np.int64)


def reference(c):
    """the result of case c: a list of columns in result order (int64 arrays, object arrays of bytes)"""
    bcode, pcode = key_codes(c)
    rows = build_passes(c)
    order = rows[np.argsort(bcode[rows], kind="stable")]
    sb = bcode[order]
    lo = np.searchsorted(sb, pcode, "left")
    hi = np.searchsorted(sb, pcode, "right")
    cnt = hi - lo
    if c.single:
        cnt = np.minimum(cnt, 1)
    if c.agg is None:
        pidx = np.repeat(np.arange(len(pcode)), cnt)
        start = np.repeat(lo, cnt)
        step = np.arange(len(pidx)) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        bidx = order[start + step]
        return [_column(c, "p", o, pidx) for o in c.out] + [_column(c, "b", v, bidx) for v in c.pay]
    # per probe tuple: matches, and the sum of its matches' payloads (prefix sums wrap around 2^64)
    pay = c.build[c.pay[0]][order].astype(np.int64).view(np.uint64)
    csum = np.concatenate([np.zeros(1, np.uint64), np.cumsum(pay, dtype=np.uint64)])
    sum_b = csum[hi] - csum[lo]
    sum_p = cnt.astype(np.uint64) * c.probe[c.pval].astype(np.int64).view(np.uint64)
    hit = cnt > 0
    if c.agg == "all":
        if not hit.any():
            return [np.zeros(0, np.int64)] * 3
        return [np.array([x.sum(dtype=np.uint64)]).view(np.int64) for x in (cnt.astype(np.uint64), sum_b, sum_p)]
    keys, g = np.unique(c.probe[c.pkeys[0]].astype(np.int64)[hit], return_inverse=True)
    out = [keys]
    for x in (cnt.astype(np.uint64), sum_b, sum_p):
        acc = np.zeros(len(keys), np.uint64)
        np.add.at(acc, g.reshape(-1), x[hit])
        out.append(acc.view(np.int64))
    return out


def canonical_rows(cols, sql):
    """result columns -> one row per tuple as a sorted list of tuples: integers as int64, strings as
    bytes (CHAR without its trailing blanks), so that two results compare as multisets"""
    canon = []
    for a, (t, w) in zip(cols, sql):
        if t == SQL_VARCHAR or (t == SQL_CHAR and w > 1):
            s = _strings(a) if a.dtype.kind == "S" else a
            canon.append(s if t == SQL_VARCHAR else np.array([x.rstrip(b" ") for x in s], dtype=object))
        else:
            canon.append(np.asarray(a).astype(np.int64))
    return canon


def assert_same_rows(got, want, sql, what):
    """got, want: result columns; the same multiset of tuples, compared as int64 matrices (string
    columns replaced by their rank among the strings of both)"""
    g, w = canonical_rows(got, sql), canonical_rows(want, sql)
    ng, nw = (len(g[0]) if g else 0), (len(w[0]) if w else 0)
    assert ng == nw, f"{what}: {ng} rows, the reference has {nw}"
    mats = [[], []]
    for x, y in zip(g, w):
        if x.dtype == object:
            inv = np.unique(np.concatenate([x, y]), return_inverse=True)[1].reshape(-1).astype(np.int64)
            x, y = inv[:ng], inv[ng:]
        mats[0].append(x)
        mats[1].append(y)
    a, b = (np.stack(m, axis=1) if m else np.zeros((0, 0), np.int64) for m in mats)
    a, b = (m[np.lexsort(m.T[::-1])] if len(m) else m for m in (a, b))
    bad = np.flatnonzero((a != b).any(axis=1)) if len(a) else []
    assert len(bad) == 0, f"{what}: {len(bad)} of {ng} sorted rows differ, first {a[bad[0]].tolist()} vs {b[bad[0]].tolist()}"
