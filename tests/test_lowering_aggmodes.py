"""CPU check of the host choices the register and shared-memory aggregation paths rely on for exactness:
the value bounds of an aggregate (upload statistics narrowed by `col CMP const` selections, interval
arithmetic), the SUM accumulation mode and flush bound chosen from them, and the packed group key.
rq_debug_lower prints the choices; they must equal the exact restatement in agg_limit_plans.py at every
edge of the rules, and the flush bound must keep every 32-bit piece sum from wrapping."""
import pytest

import agg_limit_plans as A

COLS = ["k", "v", "w", "b"]
TYPES, WIDTHS = [A.RQ_I32, A.RQ_I64, A.RQ_I64, A.RQ_I8], [4, 8, 8, 1]
K_STATS, B_STATS = (0, 3), (0, 1)


def check_modes(d, stats, expect_aggs):
    """expect_aggs: [(kind, lo, hi)] in the plan's value order, COUNT(*) last"""
    r = A.lower(d, A.IMPL_REGAGG, TYPES, WIDTHS, stats)
    assert len(r["aggmap"]) == len(expect_aggs)
    for k, (kind, lo, hi) in enumerate(expect_aggs):
        u = r["aggmap"][k][0]
        assert r["agg"][u] == (kind,)
        mode, shift, _ = A.agg_mode(kind, lo, hi)
        assert r["aggmode"][u] == (mode, shift), f"aggregate {k} over [{lo}, {hi}]"
    flush = A.flush_bound(expect_aggs)
    assert r["flushbound"] == flush
    # soundness: kR values a tile of at most piece_max each, for `flush` tiles, fit in 32 bits; and the
    # bound is the largest that does for the piece (or tuple counter) that limits it
    pieces = [p for kind, lo, hi in expect_aggs for p in A.agg_mode(kind, lo, hi)[2]] + [1]
    assert flush >= 1
    for p in pieces:
        assert A.KR * flush * p < 2 ** 32
    assert any(A.KR * (flush + 1) * max(p, 1) >= 2 ** 32 for p in pieces)
    return r


def sum_count(value, filters=(), kinds=(A.AGG_SUM,)):
    return A.sum_by(COLS, ["k"], value, filters, kinds)


EDGES = [0, 1, 2 ** 25 - 1, 2 ** 25, 2 ** 32 - 1, 2 ** 32, 2 ** 48 - 1, 2 ** 48, A.I64_MAX]


@pytest.mark.parametrize("hi", EDGES)
@pytest.mark.parametrize("lo", [0, -1, A.I64_MIN])
def test_sum_mode_at_every_edge(lo, hi):
    stats = [K_STATS, (lo, hi), (0, 1), B_STATS]
    r = check_modes(sum_count("v"), stats, [(A.AGG_SUM, lo, hi), (A.AGG_COUNT, 0, 0)])
    if lo == 0:
        expect = A.AM_P1 if hi < 2 ** 25 else A.AM_W64 if hi < 2 ** 32 else A.AM_P2 if hi < 2 ** 48 else A.AM_FULL
        assert r["aggmode"][0][0] == expect


def test_flush_bound_of_the_widest_pieces():
    """the bounds the GPU tests rely on: 16 tiles at P1's largest value, 32 at P2's"""
    assert A.flush_bound([(A.AGG_SUM, 0, 2 ** 25 - 1)]) == 16
    assert A.flush_bound([(A.AGG_SUM, 0, 2 ** 48 - 1)]) == 32
    assert A.flush_bound([(A.AGG_SUM, 0, 2 ** 32 - 1)]) == 2 ** 29 - 1


@pytest.mark.parametrize("kind", [A.AGG_MIN, A.AGG_MAX])
def test_min_max_take_the_64_bit_form(kind):
    stats = [K_STATS, (0, 5), (0, 1), B_STATS]
    check_modes(sum_count("v", kinds=(kind, A.AGG_SUM)), stats,
                [(kind, 0, 5), (A.AGG_SUM, 0, 5), (A.AGG_COUNT, 0, 0)])


def test_no_statistics_means_unknown():
    r = A.lower(sum_count("v"), A.IMPL_REGAGG, TYPES, WIDTHS, None)
    assert r["aggmode"][0] == (A.AM_FULL, 0)
    # a 4-byte column without statistics is still bounded by its type, but may be negative
    r = A.lower(sum_count("k"), A.IMPL_REGAGG, TYPES, WIDTHS, None)
    assert r["aggmode"][0] == (A.AM_FULL, 0)
    # a 1-byte column is unsigned
    r = A.lower(sum_count("b"), A.IMPL_REGAGG, TYPES, WIDTHS, None)
    assert r["aggmode"][0] == (A.AM_P1, 0) and r["flushbound"] == A.bound_tiles(255)


V_WIDE = (0, 2 ** 40)
FILTERS = [
    [("v", "LT", 2 ** 25, False)],
    [("v", "LE", 2 ** 25 - 1, False)],
    [("v", "LE", 2 ** 25, False)],
    [("v", "GT", 2 ** 25, True)],                        # 2^25 > v
    [("v", "GE", 2 ** 32 - 1, True)],                    # 2^32 - 1 >= v
    [("v", "EQ", 2 ** 25 - 1, False)],
    [("v", "EQ", 2 ** 48 - 1, True)],
    [("v", "GE", 3, False), ("v", "LE", 2 ** 32, False)],
    [("v", "LT", 5, False), ("v", "GT", 10, False)],    # contradictory: no tuple passes
    [("v", "EQ", 7, False), ("v", "EQ", 9, False)],     # contradictory
    [("v", "LT", 0, False)],                             # below the statistics
    [("v", "GT", 2 ** 41, False)],                       # above the statistics
    [("w", "LT", 2 ** 20, False)],                       # another column: no effect on v
    [("v", "LT", A.I64_MIN + 1, False)],
]


@pytest.mark.parametrize("filters", FILTERS, ids=[repr(f) for f in FILTERS])
@pytest.mark.parametrize("vlo", [0, -(2 ** 30)])
def test_filters_narrow_the_bounds(filters, vlo):
    stats = [K_STATS, (vlo, V_WIDE[1]), (0, 2 ** 60), B_STATS]
    lo, hi = A.narrow(vlo, V_WIDE[1], [(op, k, left) for c, op, k, left in filters if c == "v"])
    check_modes(sum_count("v", filters), stats, [(A.AGG_SUM, lo, hi), (A.AGG_COUNT, 0, 0)])


def test_narrowing_rule_examples():
    """spot values of the restatement itself, so that it cannot drift along with the engine"""
    assert A.narrow(0, 2 ** 40, [("LT", 2 ** 25, False)]) == (0, 2 ** 25 - 1)
    assert A.narrow(0, 2 ** 40, [("LT", 2 ** 25, True)]) == (2 ** 25 + 1, 2 ** 40)
    assert A.narrow(0, 2 ** 40, [("LT", 5, False), ("GT", 10, False)]) == (11, 11)
    assert A.narrow(0, 2 ** 40, [("LT", -3, False)]) == (-4, -4)
    assert A.sub((0, 10), (0, 3)) == (-3, 10)
    assert A.mul((-2, 3), (-5, 4)) == (-15, 12)
    assert A.add((0, A.I64_MAX), (0, 1)) == (A.I64_MIN, A.I64_MAX)


COMPUTED = {
    # name: (value builder, stats of v and w, expected bounds from the two operands' bounds)
    "mul_p1": (lambda p: p.n("MUL", p.col("v"), p.col("w")), [(0, 2 ** 12), (0, 2 ** 12)], A.mul),
    "mul_p1_edge": (lambda p: p.n("MUL", p.col("v"), p.col("w")), [(0, 2 ** 12 + 1), (0, 2 ** 13 - 1)], A.mul),
    "mul_p2": (lambda p: p.n("MUL", p.col("v"), p.col("w")), [(0, 2 ** 24 - 1), (0, 2 ** 24 - 1)], A.mul),
    "mul_neg": (lambda p: p.n("MUL", p.col("v"), p.col("w")), [(-1, 2 ** 10), (0, 2 ** 10)], A.mul),
    "mul_negneg": (lambda p: p.n("MUL", p.col("v"), p.col("w")), [(-(2 ** 10), -1), (-(2 ** 10), -1)], A.mul),
    "mul_wraps": (lambda p: p.n("MUL", p.col("v"), p.col("w")), [(0, 2 ** 32), (0, 2 ** 31)], A.mul),
    "sub_pos": (lambda p: p.n("SUB", p.col("v"), p.col("w")), [(2 ** 20, 2 ** 24), (0, 2 ** 20)], A.sub),
    "sub_neg": (lambda p: p.n("SUB", p.col("v"), p.col("w")), [(0, 2 ** 24), (0, 1)], A.sub),
    "sub_wraps": (lambda p: p.n("SUB", p.col("v"), p.col("w")), [(A.I64_MIN, 0), (0, 1)], A.sub),
    "add_edge": (lambda p: p.n("ADD", p.col("v"), p.col("w")), [(0, 2 ** 24), (0, 2 ** 24 - 1)], A.add),
    "add_wraps": (lambda p: p.n("ADD", p.col("v"), p.col("w")), [(0, A.I64_MAX), (0, 1)], A.add),
    "case": (lambda p: p.n("SELECT", p.n("LT", p.col("k"), p.const(2)), p.col("v"), p.col("w")),
             [(0, 2 ** 25 - 1), (2 ** 25, 2 ** 32 - 1)], lambda a, b: A.select(a, b)),
    "case_neg": (lambda p: p.n("SELECT", p.n("LT", p.col("k"), p.const(2)), p.col("v"), p.col("w")),
                 [(0, 7), (-1, 7)], lambda a, b: A.select(a, b)),
}


@pytest.mark.parametrize("name", sorted(COMPUTED))
def test_computed_values(name):
    build, (vs, ws), rule = COMPUTED[name]
    lo, hi = rule(vs, ws)
    check_modes(sum_count(build), [K_STATS, vs, ws, B_STATS], [(A.AGG_SUM, lo, hi), (A.AGG_COUNT, 0, 0)])


def test_three_sums_take_the_tightest_bound():
    """the flush bound is the minimum over every piece of every SUM"""
    def build(p):
        return [(p.col("k"), A.SQL_INT)], [(p.col("v"), A.AGG_SUM), (p.col("w"), A.AGG_SUM),
                                          (p.n("ADD", p.col("v"), p.col("w")), A.AGG_SUM), (None, A.AGG_COUNT)]
    d = A.agg_plan(COLS, build)
    vs, ws = (0, 2 ** 20), (0, 2 ** 46)
    check_modes(d, [K_STATS, vs, ws, B_STATS], [(A.AGG_SUM, *vs), (A.AGG_SUM, *ws), (A.AGG_SUM, *A.add(vs, ws)),
                                               (A.AGG_COUNT, 0, 0)])


# ---- packed group keys ---------------------------------------------------------------------------------
KEY_COLS = ["a", "b", "c", "v"]


def key_plan(computed=()):
    """select a, b, c, sum(v), count(*) group by a, b, c; keys named in `computed` are key + 0 * v (a slot)"""
    def build(p):
        keys = []
        for c in ("a", "b", "c"):
            n = p.col(c)
            if c in computed:
                n = p.n("ADD", n, p.n("MUL", p.col("v"), p.const(0)))
            keys.append((n, A.SQL_BIGINT))
        return keys, [(p.col("v"), A.AGG_SUM), (None, A.AGG_COUNT)]
    return A.agg_plan(KEY_COLS, build)


def one_key_plan():
    return A.agg_plan(KEY_COLS, lambda p: ([(p.col("a"), A.SQL_BIGINT)], [(p.col("v"), A.AGG_SUM), (None, A.AGG_COUNT)]))


# (bits proven from the bound) -> (lo, hi) with hi = 2^bits - 1, the largest value of that width
def top(bits):
    return 0, 2 ** bits - 1


KEY_CASES = {
    # name: (types, widths, stats of a, b, c)
    "w31": ([3, 3, 3], [8, 8, 8], [top(10), top(10), top(11)]),
    "w32": ([3, 3, 3], [8, 8, 8], [top(10), top(11), top(11)]),
    "w32_by_one": ([3, 3, 3], [8, 8, 8], [top(10), top(10), (0, 2 ** 11)]),      # 2^11 needs 12 bits
    "w64": ([3, 3, 3], [8, 8, 8], [top(20), top(22), top(22)]),
    "w65": ([3, 3, 3], [8, 8, 8], [top(21), top(22), top(22)]),
    "zero_bounds": ([3, 3, 3], [8, 8, 8], [(0, 0), (0, 1), (0, 2)]),
    "signed_i32": ([2, 3, 3], [4, 8, 8], [(-1, 5), top(3), top(4)]),
    "signed_i32_full": ([2, 2, 3], [4, 4, 8], [(A.I32_MIN, A.I32_MAX), top(31), (0, 0)]),
    "signed_i64": ([3, 3, 3], [8, 8, 8], [(-1, 0), (0, 0), (0, 0)]),
    "byte": ([1, 1, 1], [1, 1, 1], [(0, 255), (0, 127), (0, 128)]),
    "byte_and_i32": ([1, 2, 3], [1, 4, 8], [(0, 255), (0, 2 ** 23 - 1), (0, 0)]),
    "i32_top": ([2, 3, 3], [4, 8, 8], [(0, A.I32_MAX), (0, 0), (0, 0)]),
    "i64_top": ([3, 3, 3], [8, 8, 8], [(0, A.I64_MAX), (0, 0), (0, 0)]),
    "i64_62": ([3, 3, 3], [8, 8, 8], [(0, 2 ** 62), (0, 0), (0, 0)]),
}


@pytest.mark.parametrize("impl", [A.IMPL_REGAGG, A.IMPL_LOWAGG])
@pytest.mark.parametrize("computed", [(), ("b",)])
@pytest.mark.parametrize("name", sorted(KEY_CASES))
def test_packed_key_fields(name, computed, impl):
    types, widths, stats = KEY_CASES[name]
    r = A.lower(key_plan(computed), impl, types + [3], widths + [8], stats + [(0, 9)])
    fields = []
    for c, (t, w, (lo, hi)) in enumerate(zip(types, widths, stats)):
        lo, hi = A.col_bounds(t, (lo, hi))
        if "abc"[c] in computed:
            # key + 0 * v: interval arithmetic gives the key's own bounds, but the value is a slot
            lo, hi = A.add((lo, hi), A.mul((0, 9), (0, 0)))
            fields.append(A.key_field(lo, hi))
        else:
            fields.append(A.key_field(lo, hi, w))
    expect = A.pack_keys(fields)
    assert r["packed"] == int(expect is not None)
    if expect is None:
        assert "key32" not in r
        return
    layout, key32 = expect
    assert [r["keyfield"][k] for k in range(3)] == layout
    assert r["key32"] == key32


def test_key_field_widths():
    """the key-width edges the GPU tests use, in numbers"""
    assert A.pack_keys([A.key_field(*top(10), 8), A.key_field(*top(10), 8), A.key_field(*top(11), 8)])[1] == 1
    assert A.pack_keys([A.key_field(*top(10), 8), A.key_field(*top(11), 8), A.key_field(*top(11), 8)])[1] == 0
    assert A.pack_keys([A.key_field(*top(20), 8), A.key_field(*top(22), 8), A.key_field(*top(22), 8)]) is not None
    assert A.pack_keys([A.key_field(*top(21), 8), A.key_field(*top(22), 8), A.key_field(*top(22), 8)]) is None
    assert A.key_field(0, 2 ** 11, 8) == (12, 0)
    assert A.key_field(-1, 5, 4) == (32, 1)
    assert A.key_field(0, 255, 1) == (8, 0)
    assert A.key_field(0, A.I64_MAX, 8) == (63, 0)
    assert A.key_field(0, 0, 8) == (1, 0)


@pytest.mark.parametrize("stats,expect", [
    (top(31), ((0, 31, 0),)), (top(32), ((0, 32, 0),)), ((-1, 1), ((0, 64, 1),)),
    ((A.I64_MIN, A.I64_MAX), ((0, 64, 1),)), ((0, 2 ** 31), ((0, 32, 0),))])
def test_one_key(stats, expect):
    r = A.lower(one_key_plan(), A.IMPL_REGAGG, [3, 3, 3, 3], [8, 8, 8, 8], [stats, (0, 0), (0, 0), (0, 9)])
    assert tuple(r["keyfield"][k] for k in range(len(r["keyfield"]))) == expect
    assert r["key32"] == int(expect[0][1] <= 31)
