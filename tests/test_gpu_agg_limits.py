"""Grouped aggregation on the B200 at the limits its exactness rests on, against the plan oracle and, for
every SUM, an exact Python-integer sum reduced mod 2^64 (which checks the oracle's wrap-around as well):

- every SUM accumulation mode at its edge value, with every value at the bound, so that a lane's 32-bit
  piece sums end just below 2^32 before each flush, on row counts that give many flushes and a ragged
  last tile;
- bounds narrowed by selections, with the rows that fail them holding values far above the bound;
- group counts around the register path (4 a warp), the shared-memory path (8 a warp) and the global
  group table (2048), including a layout where every warp's groups fit but the table overflows;
- packed group keys at every bit-width edge;
- random plans, whose small size hints make the hash table fill and the scan drain its ring early
  (at one and at eight warps a CTA, with a ring of one stage);

each under several launch geometries (warps a CTA, TMA ring stages), read back from rq_debug_lower for
the path that runs, to make sure the geometry took effect. Which path ran is read from the engine's
trace: every overflow of a group path makes the engine rerun the pipeline with the next path, and the
trace counts these reruns."""
import contextlib
import itertools
import re

import numpy as np
import pytest

import agg_limit_plans as A
from common import plan_tables, serialize_columns, assert_same_relation
from oracle.plan_oracle import run_plan
from resql_b200 import Plan

pytestmark = pytest.mark.gpu

# (warps, stages); None: the automatic choice. 16 warps of 4 stages fit only tiles of at most 3 KB (a 4- and
# an 8-byte column); wider tables take 16 warps and 4 stages separately.
GEOMETRIES = [None, (1, 1), (1, 2), (8, 1), (16, 4)]
WIDE_GEOMETRIES = [None, (1, 1), (1, 2), (8, 1), (16, 1), (4, 4)]
N1, N2 = 2 ** 21 + 37, 2 ** 22 + 7          # many tiles a warp at warps=1, and a ragged last tile
N_GROUPS = 2 ** 20 + 3
PHYS = {np.dtype(np.int64): (A.RQ_I64, 8), np.dtype(np.int32): (A.RQ_I32, 4), np.dtype(np.uint8): (A.RQ_I8, 1)}
SQL_OF = {np.dtype(np.int64): (A.SQL_BIGINT, 0), np.dtype(np.int32): (A.SQL_INT, 0), np.dtype(np.uint8): (A.SQL_CHAR, 1)}


def key_sql(table, names):
    return {c: SQL_OF[table[c].dtype] for c in names}


@pytest.fixture(scope="module")
def engine():
    from resql_b200 import Engine
    eng = Engine(0)
    try:
        yield eng
    finally:
        for opt in ("warps", "stages", "trace"):
            eng.set_option(opt, 0)
        eng.shutdown()


@contextlib.contextmanager
def geometry(engine, geo):
    """the launch geometry geo (None: automatic), with the trace on"""
    warps, stages = geo or (0, 0)
    engine.set_option("warps", warps)
    engine.set_option("stages", stages)
    engine.set_option("trace", 1)
    try:
        yield
    finally:
        for opt in ("warps", "stages", "trace"):
            engine.set_option(opt, 0)


_TAGS = itertools.count()


def tagged(d):
    """d with a dead constant appended to every pipeline, different in every call: the engine remembers
    per pipeline which aggregation path worked and starts there next time, so without the tag a plan
    that overflowed the register path once would never run on it again in this module"""
    import copy
    d = copy.deepcopy(d)
    tag = next(_TAGS)
    for p in d["pipelines"]:
        p["nodes"].append([2, 0, 0, 0, 7_000_000 + tag])
    return d


def lowering(d, table, impl=A.IMPL_REGAGG):
    cols = [table[c] for c in d["tables"][0]["columns"]]
    types, widths = zip(*(PHYS[c.dtype] for c in cols))
    stats = [(int(c.min()), int(c.max())) for c in cols]
    return A.lower(d, impl, list(types), list(widths), stats)


def reruns(err):
    """(reruns, last reason) of the last plan execution, from the engine's trace on stderr"""
    runs = re.findall(r"careful run rc=0 clean=\d retries=(\d+) \(([^)]*)\)", err)
    assert runs, "no trace of the execution"
    return int(runs[-1][0]), runs[-1][1]


def most_groups_a_warp(tile_of_row, gid, n, warps, sms=148):
    """the most groups one warp meets when `warps` warps a CTA scan n rows: tile t goes to warp
    t mod (grid * warps), as the scan kernel hands them out"""
    if len(gid) == 0:
        return 0
    tiles = max(1, -(-n // A.TILE))
    stride = min(-(-tiles // warps), sms) * warps
    ng = int(gid.max()) + 1
    pairs = np.unique((tile_of_row % stride) * ng + gid)
    return int(np.bincount(pairs // ng).max())


def exact_sums(keys, value, mask=None):
    """{key tuple: (SUM as int64 after wrap-around, COUNT)} in Python integers"""
    if mask is not None:
        keys, value = [k[mask] for k in keys], value[mask]
    if len(value) == 0:
        return {}
    if keys:
        uniq, inv = np.unique(np.stack(keys, axis=1), axis=0, return_inverse=True)
        inv = inv.reshape(-1)
    else:
        uniq, inv = np.zeros((1, 0), np.int64), np.zeros(len(value), np.int64)
    order = np.argsort(inv, kind="stable")
    starts = np.flatnonzero(np.r_[True, np.diff(inv[order]) != 0])
    v = value.astype(np.int64)[order]
    lo = np.add.reduceat(v & 0xFFFFFFFF, starts)           # < 2^32 each, < 2^55 summed
    hi = np.add.reduceat(v >> 32, starts)
    cnt = np.diff(np.r_[starts, len(v)])
    return {tuple(int(x) for x in uniq[g]): (A.wrap64((int(hi[i]) << 32) + int(lo[i])), int(cnt[i]))
            for i, g in enumerate(inv[order][starts])}


def run_and_check(engine, d, table, handle, want, exact, what):
    """engine result == oracle (want) and, when given, == exact {key: (sum, count)} (SUM then COUNT
    are the last two values of the plan)"""
    res, _ = engine.execute(Plan(d), {"t": handle})
    got = serialize_columns(res.columns, res.sql_types, res.sql_widths)
    assert_same_relation(got, want, d, what)
    if exact is not None:
        nk = len(d["pipelines"][0]["keys"])
        rows = {tuple(int(res.columns[k][i]) for k in range(nk)): (int(res.columns[-2][i]), int(res.columns[-1][i]))
                for i in range(res.n_rows)}
        assert rows == exact, f"{what}: engine sums differ from the exact sums"


def check_geometry(d, table, geo, what):
    """the requested geometry took effect; returns the lowering as printed"""
    r = lowering(d, table)
    if geo is not None:
        assert (r["warps"], r["stages"]) == geo, f"{what}: asked for {geo}, lowered with {(r['warps'], r['stages'])}"
    return r


def run_geometries(engine, capfd, d, table, exact, what, flushes=False, geometries=GEOMETRIES, passing=None):
    """runs d under every geometry and checks its result, its geometry and the path that ran: the register
    path when no warp meets more than 4 groups and the global table holds them all, else the
    shared-memory path (one rerun) when it runs and holds them, else hash aggregation.
    passing: the rows that reach the sink (all by default)"""
    n = len(next(iter(table.values())))
    pl = d["pipelines"][0]
    key_cols = [d["tables"][0]["columns"][pl["nodes"][k[0]][1]] for k in pl["keys"]]
    rows = np.flatnonzero(passing) if passing is not None else np.arange(n)
    if key_cols:
        gid = np.unique(np.stack([table[c][rows].astype(np.int64) for c in key_cols], axis=1), axis=0,
                        return_inverse=True)[1].reshape(-1)
    else:
        gid = np.zeros(len(rows), np.int64)
    n_groups = int(gid.max()) + 1 if len(gid) else 0
    handle = engine.upload("t", table)
    try:
        want = serialize_columns(*run_plan(d, {"t": table}))
        for geo in geometries:
            with geometry(engine, geo):
                reg = check_geometry(d, table, geo, what)
                if flushes and geo is not None and geo[0] == 1:
                    assert reg["flushbound"] < A.tiles_per_warp(n, 1), f"{what}: warps=1 does not flush"
                low = lowering(d, table, A.IMPL_LOWAGG)
                G = low["lowagg_groups"]
                if not reg["packed"]:
                    path = "hash"
                elif (not key_cols or most_groups_a_warp(rows // A.TILE, gid, n, reg["warps"]) <= 4) and n_groups <= 2048:
                    path = "register"
                elif G and most_groups_a_warp(rows // A.TILE, gid, n, low["warps"]) <= G and n_groups <= 2048:
                    path = "smem"
                    if geo is not None:
                        assert (low["warps"], low["stages"]) == geo, f"{what}: the shared-memory path lowered with {(low['warps'], low['stages'])}"
                else:
                    path = "hash"
                capfd.readouterr()
                run_and_check(engine, tagged(d), table, handle, want, exact, f"{what} {geo}")
                k, why = reruns(capfd.readouterr().err)
                if path == "register":
                    assert k == 0, f"{what} {geo}: the register path should hold every group ({k} reruns, {why})"
                elif path == "smem":
                    assert (k, why) == (1, "group overflow"), f"{what} {geo}: expected one rerun, on the shared-memory path ({k}, {why})"
                elif reg["packed"]:
                    assert k >= (2 if G else 1), f"{what} {geo}: the group paths should have overflowed first ({k} reruns, {why})"
    finally:
        handle.free()


# ---- SUM accumulation modes at their edges ---------------------------------------------------------------
def mode_table(name, n):
    r = np.arange(n, dtype=np.int64)
    k = (r % 4).astype(np.int32)
    if name == "sub":                           # SUM(v - w): negative differences of non-negative columns
        return {"k": k, "v": (r % 11).astype(np.uint8), "w": (r * 7 % 11).astype(np.uint8)}
    if name == "full_mix":                      # INT64_MIN / INT64_MAX / -1 / 0: wraps in every direction
        v = np.array([A.I64_MIN, A.I64_MAX, -1, 0, A.I64_MAX, 1], np.int64)[r % 6]
    elif name == "full_max":
        v = np.full(n, A.I64_MAX, np.int64)
    elif name == "full_min":
        v = np.full(n, A.I64_MIN, np.int64)
    else:
        v = np.full(n, {"p1": 2 ** 25 - 1, "w64_low": 2 ** 25, "w64": 2 ** 32 - 1, "p2_low": 2 ** 32,
                        "p2": 2 ** 48 - 1, "full": 2 ** 48}[name], np.int64)
    v[n // 2] = 0                               # statistics lo = 0 (the full_* tables are signed anyway)
    return {"k": k, "v": v, "w": np.zeros(n, np.int64)}


MODE_CASES = [("p1", N2, A.AM_P1), ("p1", N1, A.AM_P1), ("w64_low", N1, A.AM_W64), ("w64", N2, A.AM_W64),
              ("p2_low", N1, A.AM_P2), ("p2", N2, A.AM_P2), ("p2", N1, A.AM_P2), ("full", N1, A.AM_FULL),
              ("full_max", N2, A.AM_FULL), ("full_min", N1, A.AM_FULL), ("full_mix", N2, A.AM_FULL),
              ("sub", N1, A.AM_FULL)]


@pytest.mark.parametrize("name,n,mode", MODE_CASES, ids=[f"{c}-{n}" for c, n, _ in MODE_CASES])
def test_sum_modes_at_their_edges(name, n, mode, engine, capfd):
    t = mode_table(name, n)
    if name == "sub":
        d = A.sum_by(["k", "v", "w"], ["k"], lambda p: p.n("SUB", p.col("v"), p.col("w")), key_sql=key_sql(t, ["k"]))
        value = t["v"].astype(np.int64) - t["w"]
    else:
        d = A.sum_by(["k", "v", "w"], ["k"], "v", key_sql=key_sql(t, ["k"]))
        value = t["v"]
    assert lowering(d, t)["aggmode"][0][0] == mode
    run_geometries(engine, capfd, d, t, exact_sums([t["k"].astype(np.int64)], value), f"{name}@{n}",
                   flushes=name in ("p1", "p2"))


def test_sum_without_group_by_at_the_p1_edge(engine, capfd):
    t = mode_table("p1", N2)
    d = A.sum_by(["k", "v", "w"], [], "v")
    run_geometries(engine, capfd, d, t, exact_sums([], t["v"]), "no group by", flushes=True)


# ---- bounds narrowed by selections --------------------------------------------------------------------------
FILTER_CASES = {
    # name: (passing value, failing value, filters on v, mode of the narrowed bound)
    "lt_p1": (2 ** 25 - 1, 2 ** 40, [("v", "LT", 2 ** 25, False)], A.AM_P1),
    "const_left_p1": (2 ** 25 - 1, 2 ** 62, [("v", "GT", 2 ** 25, True)], A.AM_P1),
    "eq_p2": (2 ** 48 - 1, 2 ** 60, [("v", "EQ", 2 ** 48 - 1, False)], A.AM_P2),
    "range_w64": (2 ** 32 - 1, -(2 ** 40), [("v", "GE", 0, False), ("v", "LE", 2 ** 32 - 1, False)], A.AM_W64),
    "range_p2": (2 ** 48 - 1, -(2 ** 40), [("v", "GE", 0, False), ("v", "LT", 2 ** 48, False)], A.AM_P2),
    "contradictory": (3, 2 ** 40, [("v", "LT", 5, False), ("v", "GT", 10, False)], A.AM_P1),
}


@pytest.mark.parametrize("name", sorted(FILTER_CASES))
def test_filter_narrowed_bounds(name, engine, capfd):
    good, bad, filters, mode = FILTER_CASES[name]
    n = N1
    r = np.arange(n, dtype=np.int64)
    v = np.where(r % 3 == 2, bad, good).astype(np.int64)
    k = np.where(r % 3 == 2, 2 ** 30 + 3, r % 4).astype(np.int32)      # the failing rows' keys lie far outside too
    t = {"k": k, "v": v, "w": np.zeros(n, np.int64)}
    filters = filters + [("k", "LE", 3, False)]
    d = A.sum_by(["k", "v", "w"], ["k"], "v", filters, key_sql=key_sql(t, ["k"]))
    low = lowering(d, t)
    assert low["aggmode"][0][0] == mode and low["keyfield"][0] == (0, 2, 0)
    passing = (r % 3 != 2) & (name != "contradictory")
    run_geometries(engine, capfd, d, t, exact_sums([t["k"].astype(np.int64)], v, passing), name,
                   flushes=name not in ("contradictory", "range_w64"), passing=passing)


# ---- group counts -----------------------------------------------------------------------------------------
def group_keys(g, nkeys):
    """group ids -> nkeys int64 key columns that tell the groups apart (non-negative, so that the key packs)"""
    if nkeys == 1:
        return [g.astype(np.int64)]
    return [(g % 13).astype(np.int64), (g // 13 % 17).astype(np.int64), (g // 221).astype(np.int64)]


GROUP_CASES = [(layout, groups, nkeys) for nkeys in (1, 3) for layout, groups in
               [("mod", 1), ("mod", 4), ("mod", 5), ("mod", 8), ("mod", 9), ("mod", 2048), ("mod", 2049),
                ("tile", 2048), ("tile", 2049), ("tile", 2368)]]


@pytest.mark.parametrize("layout,groups,nkeys", GROUP_CASES, ids=[f"{l}{g}-k{k}" for l, g, k in GROUP_CASES])
def test_group_counts(layout, groups, nkeys, engine, capfd):
    """mod: every warp meets every group; tile: sorted keys, one a tile, so that each warp meets only a
    few groups while the global group table (2048 slots) fills or overflows"""
    if layout == "mod":
        n = N_GROUPS
        g = np.arange(n, dtype=np.int64) % groups
    else:
        n = groups * A.TILE - 100                               # the last tile ragged
        g = np.arange(n, dtype=np.int64) // A.TILE
    keys = group_keys(g, nkeys)
    names = [f"k{i}" for i in range(nkeys)]
    t = dict(zip(names, keys))
    t["v"] = np.full(n, 2 ** 25 - 1, np.int64)
    t["v"][0] = 0
    d = A.sum_by(names + ["v"], names, "v")
    run_geometries(engine, capfd, d, t, exact_sums(keys, t["v"]), f"{layout} {groups} groups, {nkeys} keys",
                   flushes=layout == "mod" and groups <= 4, geometries=WIDE_GEOMETRIES)


# ---- packed group keys at their width edges ------------------------------------------------------------------
KEY_EDGES = {
    # name: bit widths of three keys (values 0 .. 2^b - 1), or "signed" cases with explicit values
    "w31": (10, 10, 11), "w32": (10, 11, 11), "w64": (20, 22, 22), "w65": (21, 22, 22),
    "w1": (1, 1, 1), "one63": (63,), "one32": (32,), "one31": (31,),
}
SIGNED_KEYS = {
    "i64_extremes": [np.array([A.I64_MIN, A.I64_MAX, -1, 0, 1, A.I64_MIN + 1, 2 ** 62], np.int64)],
    "i32_extremes": [np.array([A.I32_MIN, A.I32_MAX, -1, 0, 1, 7, -7], np.int32)],
    "mixed": [np.array([-1, 0, 5, -1, 5, 2, 3], np.int32), np.array([0, 2 ** 20 - 1, 1, 2 ** 20 - 1, 0, 3, 3], np.int64),
              np.array([255, 0, 128, 127, 1, 255, 0], np.uint8)],
}


def key_table(name, distinct, n):
    """n rows cycling through `distinct` key tuples at the edges of each field"""
    r = np.arange(n, dtype=np.int64) % distinct
    if name in SIGNED_KEYS:
        cols = [c[r % len(c)] for c in SIGNED_KEYS[name]]
    else:
        cols = []
        for i, b in enumerate(KEY_EDGES[name]):
            edge = np.array([2 ** b - 1, 0, 2 ** (b - 1), 2 ** b - 2 if b > 1 else 1, 1, 2 ** b - 1, 0], np.int64)
            cols.append(edge[(r + i) % len(edge)])
    return cols


@pytest.mark.parametrize("distinct", [4, 7], ids=["reg", "smem"])
@pytest.mark.parametrize("name", sorted(KEY_EDGES) + sorted(SIGNED_KEYS))
def test_packed_keys_at_width_edges(name, distinct, engine, capfd):
    """4 distinct keys take the register path, 7 the shared-memory path (where it runs, warps >= 8)"""
    n = N_GROUPS
    keys = key_table(name, distinct, n)
    names = [f"k{i}" for i in range(len(keys))]
    t = dict(zip(names, keys))
    t["v"] = (np.arange(n, dtype=np.int64) % 1000) * 3
    d = A.sum_by(names + ["v"], names, "v", key_sql=key_sql(t, names))
    low = lowering(d, t)
    fields = [A.key_field(int(c.min()), int(c.max()), c.dtype.itemsize) for c in keys]
    packed = A.pack_keys(fields)
    assert low["packed"] == int(packed is not None)
    if packed is not None:
        assert [low["keyfield"][i] for i in range(len(keys))] == packed[0]
    run_geometries(engine, capfd, d, t, exact_sums([k.astype(np.int64) for k in keys], t["v"]), name,
                   geometries=WIDE_GEOMETRIES)


# ---- random plans ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sf005(engine):
    from plan_fuzz import COLS
    from resql_b200 import tpch
    data = tpch.generate(0.05, seed=5)
    up = {t: engine.upload(t, {c: data[t][c] for c, _ in cols}) for t, cols in COLS.items()}
    try:
        yield data, up
    finally:
        for h in up.values():
            h.free()


@pytest.mark.parametrize("seed", range(80))
def test_random_plans_under_small_geometries(seed, sf005, engine):
    from plan_fuzz import random_plan
    data, up = sf005
    d = random_plan(seed)
    tabs = plan_tables(d, data)
    try:
        want = serialize_columns(*run_plan(d, tabs))
    except ZeroDivisionError:
        pytest.skip("plan divides by zero")
    for geo in [(1, 1), (8, 1)]:
        with geometry(engine, geo):
            res, _ = engine.execute(Plan(tagged(d)), {t["name"]: up[t["name"]] for t in d["tables"]})
            got = serialize_columns(res.columns, res.sql_types, res.sql_widths)
            assert_same_relation(got, want, d, f"random plan {seed} {geo}")
