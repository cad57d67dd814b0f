"""Equi-joins on the B200 over adversarial key distributions, key types and run-time table forms, against
an exact reference of their own (join_key_plans.reference: sort the build keys, search the probe keys),
which a CPU test pins to the plan oracle on small instances of every case.

A join build takes one of several forms while the query runs (engine_exec.inl run_hash_sink): the
direct-address form when the key's bounds are dense enough (rerun in the hash form when a duplicate key
turns up), the hash form on one integer key (Fibonacci hash, runs that wrap from the last slot to slot
0), the hash form on composite or string keys, a table that fills and is regrown; and a probe that
meets several entries reruns in the expanded two-pass form. Every case names the form it must take,
and the engine's trace of the first (careful) execution is checked for it: one `hash table allocated +
cleared` line per hash-form attempt of the build, a `rerun (...)` line per fallback. Every case runs
with direct-address joins on and off, with the two-pass probe split forced and not, specialized and
(on a subset) interpreted, five times each: careful, replayed, captured and graph executions must all
give the reference's result."""
import itertools
import re
import zlib
from functools import lru_cache

import numpy as np
import pytest

import join_key_plans as J
from agg_limit_plans import narrow as narrowed_bounds
from common import serialize_columns, assert_same_relation
from oracle.plan_oracle import run_plan

I64 = np.int64


def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


def _wide(rng, n):
    """n payload values over the whole int64 range (their sums wrap)"""
    return rng.integers(J.I64_MIN, J.I64_MAX, n, dtype=I64, endpoint=True)


def _int_case(name, bk, pk, rng, **kw):
    """one integer key: build (bk, id), probe (pk, pid, v); materializes (pid, pk, id) unless agg"""
    build = {"bk": bk, "id": _wide(rng, len(bk))}
    probe = {"pk": pk, "pid": np.arange(len(pk), dtype=I64), "v": _wide(rng, len(pk))}
    kw.setdefault("out", ["pid", "pk"])
    return J.JoinCase(name, build, probe, ["bk"], ["pk"], kw.pop("pay", ["id"]), pval="v", **kw)


def _mix(rng, *parts):
    return rng.permutation(np.concatenate([np.asarray(p, I64) for p in parts]))


# ---- single integer key -------------------------------------------------------------------------------------
def dense_unique(name, n):
    rng = _rng(name)
    return _int_case(name, 1000 + rng.permutation(n).astype(I64), rng.integers(990, n + 1010, 2 * n, dtype=I64), rng,
                     single=1, path="direct")


def dense_one_dup(name, n):
    rng = _rng(name)
    bk = 1000 + rng.permutation(n).astype(I64)
    bk[-1] = bk[0]
    pk = rng.integers(990, n + 1010, 2 * n, dtype=I64)
    pk[:5] = bk[0]
    return _int_case(name, bk, pk, rng, path="dup", expand=True)


def sparse_unique(name, n):
    rng = _rng(name)
    bk = rng.choice(200 * n, n, replace=False).astype(I64)
    pk = _mix(rng, bk[rng.integers(0, n, n)], rng.integers(0, 200 * n, n), [bk.min(), bk.max()])
    return _int_case(name, bk, pk, rng, single=1, path="hash")


def all_negative(name, n):
    rng = _rng(name)
    return _int_case(name, -7 - rng.permutation(n).astype(I64), rng.integers(-n - 20, 5, 2 * n, dtype=I64), rng,
                     single=1, path="direct")


def _half(name, n, lo, path):
    """dense unique keys from lo up, probed from lo - 3 to the top + 3"""
    rng = _rng(name)
    bk = np.int64(lo) + rng.permutation(n).astype(I64)
    pk = np.int64(lo) + rng.integers(-3, n + 3, 2 * n, dtype=I64)
    return _int_case(name, bk, pk, rng, single=1, path=path)


def near_half_min(name, n):                 # lowest key INT64_MIN / 2 + 1: the direct form applies
    return _half(name, n, J.HALF_MIN + 1, "direct")


def at_half_min(name, n):                   # lowest key INT64_MIN / 2: it does not
    return _half(name, n, J.HALF_MIN, "hash")


def near_half_max(name, n):                 # highest key INT64_MAX / 2 - 1
    return _half(name, n, J.HALF_MAX - n, "direct")


def at_half_max(name, n):                   # highest key INT64_MAX / 2
    return _half(name, n, J.HALF_MAX - n + 1, "hash")


def int64_extremes(name, n):
    rng = _rng(name)
    edge = np.array([J.I64_MIN, J.I64_MAX, -1, 0, J.I64_MIN + 1, J.I64_MAX - 1, 1], I64)
    rest = np.setdiff1d(_wide(rng, n), edge)
    bk = _mix(rng, edge, rest)
    pk = _mix(rng, edge, edge, bk[rng.integers(0, len(bk), n)], _wide(rng, n), [2, -2])
    return _int_case(name, bk, pk, rng, single=1, path="hash")


# ---- direct-address domain edges ------------------------------------------------------------------------------
def _domain(name, n, span, path):
    """n unique keys over exactly `span` values from -12345 (both ends present); the probe keys reach
    one beyond either end, so that the build is not pruned to a narrower range"""
    rng = _rng(name)
    inner = 1 + rng.choice(span - 2, n - 2, replace=False)
    bk = _mix(rng, [0, span - 1], inner) - 12345
    pk = _mix(rng, bk[rng.integers(0, n, n)], rng.integers(-3, span + 3, n) - 12345, [-12346, span - 12345])
    return _int_case(name, bk, pk, rng, single=1, path=path)


def domain_64x(name, n):
    return _domain(name, n, 64 * n, "direct")


def domain_64x_plus_1(name, n):
    return _domain(name, n, 64 * n + 1, "hash")


FILTERS = {
    "gt_le": [("bk", "GT", 99, False), ("bk", "LE", 5000, False)],
    "const_left_ge_lt": [("bk", "LE", -500, True), ("bk", "GT", 6000, True)],       # -500 <= bk, 6000 > bk
    "lt_ge": [("bk", "LT", 4321, False), ("bk", "GE", -1000, False)],
    "eq": [("bk", "EQ", 777, False)],
    "const_left_eq": [("bk", "EQ", -3, True)],
    "contradictory": [("bk", "LT", 5, False), ("bk", "GT", 10, False)],
}


def _filtered(name, n):
    """dense unique keys over [-1000, n - 1000) under build-side selections; the probe keys take every
    value around the domain, and each end of the narrowed domain and its outside neighbours 100 times"""
    rng = _rng(name)
    filters = FILTERS[name.split("filter_", 1)[1]]
    bk = rng.permutation(n).astype(I64) - 1000
    lo, hi = narrowed_bounds(int(bk.min()), int(bk.max()), [(op, k, left) for _, op, k, left in filters])
    pk = _mix(rng, rng.integers(-1100, n - 900, 2 * n), np.repeat([lo - 1, lo, hi, hi + 1], 100))
    return _int_case(name, bk, pk, rng, single=1, filters=filters, path="direct")


# ---- a run that wraps from the last slot to slot 0 --------------------------------------------------------------
TOP26 = (2 ** 26 - 1) << 38          # a hash with its top 26 bits set: home slot last for 2^12 .. 2^26 slots


def wrap_keys(rng, m):
    """m distinct int64 keys whose hashes have their top 26 bits set"""
    low = rng.choice(2 ** 38, m, replace=False)
    return np.array([J.key_of_hash(TOP26 | int(x)) for x in low], I64)


def _wrap_dups(name, n, agg):
    rng = _rng(name)
    w = wrap_keys(rng, 1)[0]
    dups = max(300, min(3000, n // 30))
    filler = np.setdiff1d(_wide(rng, n), [w])
    bk = _mix(rng, filler, np.full(dups, w))
    pk = _mix(rng, np.full(64, w), filler[rng.integers(0, len(filler), n)], _wide(rng, n // 4))
    return _int_case(name, bk, pk, rng, agg=agg, out=["pid"], path="hash", expand=True)


def wrap_dups_count(name, n):
    return _wrap_dups(name, n, "all")


def wrap_dups_by_key(name, n):
    return _wrap_dups(name, n, "by_key")


def wrap_dups_rows(name, n):
    return _wrap_dups(name, n, None)


def wrap_unique(name, n):
    """3000 distinct keys sharing the last slot as their home: one run of 3000 that wraps"""
    rng = _rng(name)
    ws = wrap_keys(rng, max(300, min(3000, n // 30)))
    filler = np.setdiff1d(_wide(rng, n), ws)
    bk = _mix(rng, filler, ws)
    pk = _mix(rng, ws, ws[::7], filler[rng.integers(0, len(filler), n)], _wide(rng, n // 4))
    return _int_case(name, bk, pk, rng, single=1, path="hash")


# ---- mixed key widths ---------------------------------------------------------------------------------------------
def int_build_bigint_probe(name, n):
    """INT build keys (negative too) probed by BIGINT keys, some of them 2^32 away from a build key"""
    rng = _rng(name)
    bk = (rng.permutation(n) - n // 2).astype(np.int32)
    near = rng.integers(-n // 2 - 5, n // 2 + 5, 2 * n, dtype=I64)
    pk = _mix(rng, near, near[:n // 4] + 2 ** 32, near[:n // 4] - 2 ** 32)
    return _int_case(name, bk, pk, rng, single=1, path="direct")


def bigint_build_int_probe(name, n):
    """BIGINT build keys, some of them 2^32 away from an INT probe key that has no build match"""
    rng = _rng(name)
    base = (rng.permutation(n) - n // 2).astype(I64)
    bk = _mix(rng, base[n // 5:], base[:n // 10] + 2 ** 32, base[n // 10:n // 5] - 2 ** 32)
    pk = rng.integers(-n // 2 - 5, n // 2 + 5, 2 * n).astype(np.int32)
    # (the build is pruned to the probe keys' range, which leaves a dense unique domain)
    return _int_case(name, bk, pk, rng, single=1, path="direct")


def _one_byte(name, n, narrow):
    """keys that fit one byte on both sides (int64 columns: narrowed to one byte on upload, or not),
    many duplicates on the build side"""
    rng = _rng(name)
    c = _int_case(name, rng.integers(0, 251, n, dtype=I64), rng.integers(0, 256, 2 * n, dtype=I64), rng,
                  agg="by_key", path="dup", expand=True)
    c.narrow = narrow
    return c


def one_byte_narrowed(name, n):
    return _one_byte(name, n, True)


def one_byte_wide(name, n):
    return _one_byte(name, n, False)


def one_byte_unique(name, n):
    rng = _rng(name)
    c = _int_case(name, rng.permutation(251).astype(I64), rng.integers(0, 256, 2 * n, dtype=I64), rng,
                  single=1, path="direct")
    c.narrow = True
    return c


# ---- string and composite keys ------------------------------------------------------------------------------------
def _s(words, width):
    return np.array(words, dtype=f"S{width + 1}")


def _char_words(rng, n):
    """distinct words (after trailing blanks are stripped), blank-padded at random; '' and two words
    equal in their first 8 bytes among them"""
    base = [b"K%06d" % i for i in range(n)] + [b"", b"ABCDEFGH1", b"ABCDEFGH2", b"A B"]
    return [w + b" " * int(rng.integers(0, 3)) if len(w) < 10 else w for w in base]


def char_blanks(name, n):
    rng = _rng(name)
    words = _char_words(rng, n)
    probe = [words[i].rstrip(b" ") + b" " * int(rng.integers(0, 4)) for i in rng.integers(0, len(words), 2 * n)]
    probe += [b"   ", b"", b"ABCDEFGH1  ", b"ABCDEFGH3", b"ABCDEFGH", b"A B ", b"A  B", b"Z"]
    build = {"bs": _s(words, 12), "id": _wide(rng, len(words))}
    pr = {"ps": _s(probe, 12), "pid": np.arange(len(probe), dtype=I64)}
    return J.JoinCase(name, build, pr, ["bs"], ["ps"], ["id", "bs"], out=["pid", "ps"], single=1, path="hash")


def varchar_blanks(name, n):
    """trailing blanks count: 'K..' and 'K.. ' are different keys, '' and ' ' too"""
    rng = _rng(name)
    words = sorted(set(_char_words(rng, n)) | {b"K000001", b"K000001 ", b" ", b""})
    probe = [words[i] for i in rng.integers(0, len(words), 2 * n)] + [b"K000002 ", b"  ", b"ABCDEFGH1 ", b"ABCDEFGH"]
    build = {"bs": _s(words, 12), "id": _wide(rng, len(words))}
    pr = {"ps": _s(probe, 12), "pid": np.arange(len(probe), dtype=I64)}
    return J.JoinCase(name, build, pr, ["bs"], ["ps"], ["id", "bs"], out=["pid", "ps"], single=1, varchar=True, path="hash")


def int_char(name, n):
    """(INT, CHAR(6)) keys; the CHAR part blank-padded at random on either side"""
    rng = _rng(name)
    i = np.arange(n)
    a = (i % 1000 - 500).astype(np.int32)
    s = [b"S%04d" % (j // 1000) + b" " * int(rng.integers(0, 2)) for j in i]
    pick = rng.integers(0, n, 2 * n)
    pa = a[pick].copy()
    pa[::9] += 1                                            # the same string, the neighbouring int
    ps = [s[j].rstrip(b" ") + b" " * int(rng.integers(0, 2)) for j in pick]
    build = {"ba": a, "bs": _s(s, 6), "id": _wide(rng, n)}
    pr = {"pa": pa, "ps": _s(ps, 6), "pid": np.arange(2 * n, dtype=I64)}
    return J.JoinCase(name, build, pr, ["ba", "bs"], ["pa", "ps"], ["id", "bs"], out=["pid"], single=1, path="hash")


def int_int_equal_sums(name, n):
    """(a, b) keys that all sum to 7 (or 8); probes swap the parts or move one unit between them"""
    rng = _rng(name)
    a = (np.arange(n) - n // 2).astype(I64)
    b = np.where(np.arange(n) % 2 == 0, 7, 8) - a
    pick = rng.integers(0, n, 2 * n)
    pa, pb = a[pick].copy(), b[pick].copy()
    sw = slice(0, None, 5)
    pa[sw], pb[sw] = b[pick][sw], a[pick][sw]
    pa[1::7] += 1
    pb[1::7] -= 1
    build = {"ba": a, "bb": b, "id": _wide(rng, n)}
    pr = {"pa": pa, "pb": pb, "pid": np.arange(2 * n, dtype=I64)}
    return J.JoinCase(name, build, pr, ["ba", "bb"], ["pa", "pb"], ["id"], out=["pid", "pa"], single=1, path="hash")


EIGHT = [np.int64, np.int32, np.uint8, np.int64, np.int32, np.int64, np.uint8, np.int64]


def eight_keys(name, n):
    """kMaxKeys (8) key columns of three widths; each probe tuple equals a build tuple or differs from
    one in one component"""
    rng = _rng(name)
    i = np.arange(n, dtype=I64)
    parts = [i % 7, i // 7 % 5, i // 35 % 3, i // 105, -(i % 11), i % 13 - 6, (i * 7) % 256, i % 2]
    cols = [p.astype(t) for p, t in zip(parts, EIGHT)]
    pick = rng.integers(0, n, 2 * n)
    pcols = [c[pick].copy() for c in cols]
    j = rng.integers(0, 8, 2 * n)
    for k in range(8):
        m = (j == k) & (np.arange(2 * n) % 3 == 0)
        pcols[k][m] = (pcols[k][m].astype(I64) + 1).astype(EIGHT[k])
    build = {f"b{k}": c for k, c in enumerate(cols)}
    build["id"] = _wide(rng, n)
    pr = {f"p{k}": c for k, c in enumerate(pcols)}
    pr["pid"] = np.arange(2 * n, dtype=I64)
    return J.JoinCase(name, build, pr, [f"b{k}" for k in range(8)], [f"p{k}" for k in range(8)], ["id", "b2"],
                      out=["pid"], single=1, path="hash")


# ---- payloads -------------------------------------------------------------------------------------------------------
def payload_repeats_key(name, n):
    rng = _rng(name)
    c = dense_unique(name, n)
    c.build["w32"] = rng.integers(-2 ** 31, 2 ** 31, n).astype(np.int32)
    c.pay = ["bk", "id", "w32", "bk"]
    return c


def mixed_payloads(name, n):
    rng = _rng(name)
    c = dense_unique(name, n)
    c.build["w32"] = rng.integers(-2 ** 31, 2 ** 31, n).astype(np.int32)
    c.build["w8"] = rng.integers(0, 256, n).astype(np.uint8)
    c.build["s7"] = _s([b"P%d" % x + b" " * (x % 3) for x in rng.integers(0, 10 ** 4, n)], 7)
    c.pay = ["w32", "w8", "s7", "id"]
    return c


# ---- table growth -----------------------------------------------------------------------------------------------------
def grow_from_hint(name, n):
    """a size hint of 1 on a hash-form build of n rows: the table fills and is regrown"""
    rng = _rng(name)
    bk = rng.choice(300 * n, n, replace=False).astype(I64)
    pk = _mix(rng, bk[rng.integers(0, n, n)], rng.integers(0, 300 * n, n // 2), [bk.min(), bk.max()])
    return _int_case(name, bk, pk, rng, agg="all", single=1, size_hint=1, path="grow")


# ---- multi-match --------------------------------------------------------------------------------------------------------
def _multi_build(rng, n):
    """keys with 1 (most), 2 or 1000 entries each"""
    ones = np.arange(n // 2, dtype=I64)
    twos = np.arange(n // 2, n // 2 + n // 8, dtype=I64)
    thousands = np.arange(-5, 0, dtype=I64)
    return ones, twos, thousands, _mix(rng, ones, twos, twos, np.repeat(thousands, 1000))


def multi_one_pass(name, n):
    """duplicate build keys, but no probe tuple meets more than one entry: no expansion"""
    rng = _rng(name)
    ones, twos, thousands, bk = _multi_build(rng, n)
    pk = _mix(rng, ones[rng.integers(0, len(ones), 2 * n)], rng.integers(10 ** 6, 2 * 10 ** 6, n // 4))
    return _int_case(name, bk, pk, rng, path="dup")


def _multi_expand(name, n, agg):
    rng = _rng(name)
    ones, twos, thousands, bk = _multi_build(rng, n)
    pk = _mix(rng, ones[rng.integers(0, len(ones), n)], twos[rng.integers(0, len(twos), n)],
              np.repeat(thousands, max(2, n // 500)), rng.integers(10 ** 6, 2 * 10 ** 6, n // 4))
    return _int_case(name, bk, pk, rng, agg=agg, path="dup", expand=True)


def multi_expand_rows(name, n):
    return _multi_expand(name, n, None)


def multi_expand_by_key(name, n):
    return _multi_expand(name, n, "by_key")


# name: (builder, build rows on the GPU, interpreted too)
CASES = {
    "dense_unique": (dense_unique, 200_000, True),
    "dense_one_dup": (dense_one_dup, 200_000, True),
    "sparse_unique": (sparse_unique, 200_000, True),
    "all_negative": (all_negative, 100_000, False),
    "near_half_min": (near_half_min, 100_000, False),
    "at_half_min": (at_half_min, 100_000, False),
    "near_half_max": (near_half_max, 100_000, False),
    "at_half_max": (at_half_max, 100_000, False),
    "int64_extremes": (int64_extremes, 100_000, True),
    "domain_64x": (domain_64x, 16_384, False),
    "domain_64x_plus_1": (domain_64x_plus_1, 16_384, False),
    **{f"filter_{f}": (_filtered, 50_000, f == "gt_le") for f in FILTERS},
    "wrap_dups_count": (wrap_dups_count, 200_000, True),
    "wrap_dups_by_key": (wrap_dups_by_key, 200_000, False),
    "wrap_dups_rows": (wrap_dups_rows, 200_000, False),
    "wrap_unique": (wrap_unique, 200_000, True),
    "int_build_bigint_probe": (int_build_bigint_probe, 100_000, True),
    "bigint_build_int_probe": (bigint_build_int_probe, 100_000, False),
    "one_byte_narrowed": (one_byte_narrowed, 100_000, False),
    "one_byte_wide": (one_byte_wide, 100_000, False),
    "one_byte_unique": (one_byte_unique, 100_000, False),
    "char_blanks": (char_blanks, 30_000, True),
    "varchar_blanks": (varchar_blanks, 30_000, False),
    "int_char": (int_char, 30_000, True),
    "int_int_equal_sums": (int_int_equal_sums, 100_000, False),
    "eight_keys": (eight_keys, 50_000, True),
    "payload_repeats_key": (payload_repeats_key, 100_000, True),
    "mixed_payloads": (mixed_payloads, 100_000, False),
    "grow_from_hint": (grow_from_hint, 1_000_000, False),
    "multi_one_pass": (multi_one_pass, 100_000, True),
    "multi_expand_rows": (multi_expand_rows, 100_000, True),
    "multi_expand_by_key": (multi_expand_by_key, 100_000, False),
}
SMALL = 4096          # build rows of the instances the oracle checks


def make(name, n):
    return CASES[name][0](name, n)


# ---- CPU: the reference against the plan oracle ---------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(CASES))
def test_reference_matches_the_oracle(name):
    c = make(name, SMALL)
    d = J.join_plan(c)
    want = serialize_columns(*run_plan(d, {"b": c.build, "p": c.probe}))
    sql = J.result_sql(c)
    ref = J.reference(c)
    assert_same_relation(serialize_columns(ref, [t for t, _ in sql], [w for _, w in sql]), want, d, name)
    assert len(want) > 0 or name == "filter_contradictory", f"{name}: the join is empty"


def test_reference_is_not_the_oracle():
    """the comparison above would notice a reference that dropped one match"""
    c = make("multi_expand_rows", SMALL)
    ref = J.reference(c)
    short = [col[1:] for col in ref]
    with pytest.raises(AssertionError):
        J.assert_same_rows(short, ref, J.result_sql(c), "short")
    J.assert_same_rows(ref, [col[::-1] for col in ref], J.result_sql(c), "reversed")


@pytest.mark.parametrize("name", ["wrap_dups_count", "wrap_unique"])
def test_wrapping_keys_live_in_the_last_slot(name):
    c = make(name, CASES[name][1])
    keys, counts = np.unique(c.build["bk"], return_counts=True)
    ws = [int(k) for k in keys[counts > 1]] if name == "wrap_dups_count" else \
        [int(k) for k in wrap_keys(_rng(name), max(300, min(3000, CASES[name][1] // 30)))]
    assert len(ws) >= 1 and all(int(k) in set(keys.tolist()) for k in ws)
    for lg in range(12, 27):
        for k in ws:
            assert J.home_slot(k, 2 ** lg) == 2 ** lg - 1, f"key {k}: home slot in a table of 2^{lg}"
    # the run is longer than kLongRun (1024) and the hash-form table is one of those capacities
    n = len(c.build["bk"])
    cap = 4096
    while cap < 3 * n:
        cap <<= 1
    assert 2 ** 12 <= cap <= 2 ** 26
    assert (counts.max() if name == "wrap_dups_count" else len(ws)) > 1024 + 1


# ---- GPU ------------------------------------------------------------------------------------------------------------
OPTIONS = {"direct_joins": 1, "split_min_rows": -1, "split_frac": -1, "specialize": 1, "trace": 0, "narrow": 1,
           "up_chunk_krows": 512, "up_threads": 0}


@pytest.fixture(scope="module")
def engine():
    from resql_b200 import Engine
    eng = Engine(0)
    try:
        yield eng
    finally:
        for k, v in OPTIONS.items():
            eng.set_option(k, v)
        eng.shutdown()


@lru_cache(maxsize=4)
def case_and_want(name):
    c = make(name, CASES[name][1])
    return c, J.reference(c)


_TAGS = itertools.count(1)


def upload(engine, capfd, c):
    """b and p on the device; a case with `narrow` set uploads its one-byte key columns narrowed
    (small upload chunks, so that tables of this size qualify) or not, and checks that they were"""
    narrow = getattr(c, "narrow", None)
    if narrow is None:
        return {"b": engine.upload("b", c.build), "p": engine.upload("p", c.probe)}
    try:
        engine.set_option("narrow", int(narrow))
        engine.set_option("up_chunk_krows", 1)
        engine.set_option("up_threads", 8)
        engine.set_option("trace", 1)
        capfd.readouterr()
        h = {"p": engine.upload("p", c.probe), "b": engine.upload("b", c.build)}
        got = re.findall(r"upload (\w): \d+ rows, (\d+) of \d+ columns narrowed", capfd.readouterr().err)
    finally:
        for k in ("narrow", "up_chunk_krows", "up_threads", "trace"):
            engine.set_option(k, OPTIONS[k])
    if narrow:
        assert any(t == "p" and int(k) >= 1 for t, k in got), f"{c.name}: the probe table was not narrowed ({got})"
    else:
        assert not got, f"{c.name}: narrowed with narrowing off ({got})"
    return h


def careful_trace(err):
    """(hash-form build attempts, reruns in order) of the careful execution traced in err"""
    allocs = len(re.findall(r"hash table allocated \+ cleared 0$", err, re.M))
    return allocs, re.findall(r"\[rq\] rerun \(([^)]*)\)", err)


DUP, REGROWN, EXPAND = "direct-address build met duplicate keys", "hash table regrown", "multi-match expansion"


def check_path(c, direct, err):
    path = c.path if direct or c.path == "grow" else "hash"
    allocs, reruns = careful_trace(err)
    assert re.search(r"careful run rc=0", err), f"{c.name}: no trace of a careful execution"
    what = f"{c.name} (direct_joins={direct}): {allocs} hash-form builds, reruns {reruns}"
    if path == "direct":
        assert allocs == 0, what
    elif path in ("hash", "dup"):
        assert allocs == 1, what
    else:
        assert allocs >= 2, what
    assert reruns.count(DUP) == (path == "dup"), what
    assert (REGROWN in reruns) == (path == "grow"), what
    assert (EXPAND in reruns) == c.expand, what


def execute_five_times(engine, capfd, c, want, direct, split, spec, handles=None, tag=None):
    """runs case c under the given options: careful (traced), careful or replayed, replayed,
    captured, graph; every result must be the reference's. Returns the careful run's trace."""
    from resql_b200 import Plan
    sql = J.result_sql(c)
    plan = Plan(J.join_plan(c, next(_TAGS) if tag is None else tag))
    own = handles is None
    h = upload(engine, capfd, c) if own else handles
    try:
        engine.set_option("direct_joins", direct)
        engine.set_option("split_min_rows", 0 if split else -1)
        engine.set_option("split_frac", 1e18 if split else -1)
        engine.set_option("specialize", spec)
        results = []
        for run in range(5):
            engine.set_option("trace", int(run == 0))
            capfd.readouterr()
            res, _ = engine.execute(plan, h)
            if run == 0:
                err = capfd.readouterr().err
            results.append(res)
        engine.set_option("trace", 0)
    finally:
        for k, v in OPTIONS.items():
            engine.set_option(k, v)
        if own:
            for t in h.values():
                t.free()
    what = f"{c.name} direct_joins={direct} split={split} specialize={spec}"
    for run, res in enumerate(results):
        J.assert_same_rows(res.columns, want, sql, f"{what} execution {run + 1}")
    if len(want[0]) <= 50_000:
        got = serialize_columns(results[0].columns, results[0].sql_types, results[0].sql_widths)
        assert_same_relation(got, serialize_columns(want, [t for t, _ in sql], [w for _, w in sql]), plan.d, what)
    return err


GPU_RUNS = [(name, direct, split, 1) for name in CASES for direct in (1, 0) for split in (0, 1)] + \
           [(name, 1, 0, 0) for name in CASES if CASES[name][2]]


@pytest.mark.gpu
@pytest.mark.parametrize("name,direct,split,spec", GPU_RUNS,
                         ids=[f"{n}-direct{d}-split{s}-spec{p}" for n, d, s, p in GPU_RUNS])
def test_join_keys(name, direct, split, spec, engine, capfd):
    c, want = case_and_want(name)
    err = execute_five_times(engine, capfd, c, want, direct, split, spec)
    check_path(c, direct, err)


@pytest.mark.gpu
def test_capacity_memo_too_small(engine, capfd):
    """the same plan on a new upload with as many rows, ten times as many of them passing the build's
    selection (and as many more distinct keys): the capacity remembered from the first is too small"""
    n = 1_000_000
    rng = _rng("capacity_memo")
    bk = rng.choice(300 * n, n, replace=False).astype(I64)
    pk = _mix(rng, bk[rng.integers(0, n, n)], rng.integers(0, 300 * n, n // 2), [bk.min(), bk.max()])
    first = _int_case("memo_first", bk, pk, rng, agg="all", single=1, filters=[("f", "EQ", 1, False)], path="hash")
    first.build["f"] = (np.arange(n) % 10 == 0).astype(np.uint8)
    second = J.JoinCase("memo_second", dict(first.build, f=np.ones(n, np.uint8)), first.probe, ["bk"], ["pk"], ["id"],
                        agg="all", pval="v", single=1, filters=first.filters, path="grow")
    tag = next(_TAGS)
    for c in (first, second):
        err = execute_five_times(engine, capfd, c, J.reference(c), 1, 0, 1, tag=tag)
        check_path(c, 1, err)
