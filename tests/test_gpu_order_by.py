"""ORDER BY ... LIMIT on the B200 over adversarial keys, types, ties and row counts, against an exact
reference of its own (order_plans.reference), which test_order_plans.py pins to the plan oracle on
small instances of every case here.

The engine orders a final relation of n rows on one of three paths (engine_exec.inl
order_permutation): one bitonic sort in a CTA (n <= 4096); an LSD radix sort over order-preserving
64-bit keys (a string key is one key per 8 bytes of its declared width) that skips the 4-bit digits
no key varies in; and, for LIMIT k <= 2048, a radix select of the k-th first-key value that keeps the
rows up to it, ties included, and sorts those - or falls back to the radix sort when more than 4096
rows are candidates. Every case names the path it must take, and the engine's trace of the first
(careful) execution is checked for it (`[rq] order by: ...`): the path, the digit passes of a radix
sort where the case fixes them, and the exact candidate count of a radix select. Every case runs
five times (careful, replayed, captured and twice from the graph); the top-k cases run again with
the radix select off, a subset runs interpreted, and the results of all executions must be ones the
reference allows (assert_ordered_equal).

A recorded plan predicts the host's reads of device values (the varying-bits mask of every radix key
word, the candidate count of a radix select). A new upload is a new table to the engine, so these
predictions only go stale when a borrowed table's memory changes under the same handle; the last
tests do that and check that the stale prediction is noticed and the plan reruns the careful way."""
import itertools
import re
import zlib
from functools import lru_cache

import numpy as np
import pytest

import order_plans as O
from order_plans import OrderCase, SQL_VARCHAR, SQL_BOOL, SQL_DECIMAL, SQL_DATE, AGG_SUM, AGG_COUNT, AGG_MIN, AGG_MAX

pytestmark = pytest.mark.gpu

I64 = np.int64
BITONIC_MAX, TOPK_MAX = 4096, 2048
RQ_ERR_INVALID, RQ_ERR_UNSUPPORTED = 1, 3


def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


def _wide(rng, n):
    return rng.integers(O.I64_MIN, O.I64_MAX, n, dtype=I64, endpoint=True)


def _ids(n):
    return np.arange(n, dtype=I64)


def path_of(n, limit, topk=True):
    """the path the engine takes for n rows unless a radix select falls back"""
    if n <= 1:
        return "none"
    if n <= BITONIC_MAX:
        return "bitonic"
    return "topk" if topk and 0 <= limit <= TOPK_MAX else "radix"


# ---- row counts ---------------------------------------------------------------------------------------------
EDGES = np.array([O.I64_MIN, O.I64_MIN + 1, -1, 0, 1, O.I64_MAX - 1, O.I64_MAX], I64)
SIZES = [0, 1, 2, 3, 255, 256, 257, 4095, 4096, 4097, 6143, 6144, 6145, 100_003, 2_000_000]


def bigint_keys(rng, n):
    """n BIGINT keys over the whole range, the int64 edges among them, one in 8 a repeat"""
    k = _wide(rng, n)
    k[rng.integers(0, n, n // 8)] = k[rng.integers(0, n, n // 8)] if n else k[:0]
    m = min(n, len(EDGES))
    k[rng.choice(n, m, replace=False)] = EDGES[:m] if n < len(EDGES) else EDGES
    return k


def sized(name, n, asc=True, passes=None):
    rng = _rng(name)
    t = {"k": bigint_keys(rng, n), "id": _ids(n)}
    return OrderCase(name, t, ["k", "id"], [(0, asc)], path=path_of(n, -1), passes=passes)


# ---- key types ----------------------------------------------------------------------------------------------------
def typed(name, n, kind, asc):
    """one key of a type (its extremes among random values, one in 4 a repeat) and a row id"""
    rng = _rng(name)
    sql = {}
    if kind == "bigint":
        k = bigint_keys(rng, n)
    elif kind in ("int", "date"):
        k = rng.integers(O.I32_MIN, O.I32_MAX, n, dtype=I64, endpoint=True)
        k[:6] = [O.I32_MIN, O.I32_MIN + 1, -1, 0, O.I32_MAX - 1, O.I32_MAX]
        k = k.astype(np.int32)
        if kind == "date":
            sql["k"] = (SQL_DATE, 0)
    elif kind == "decimal":                                # DECIMAL(15,2), mostly negative
        k = rng.integers(-10 ** 15, 10 ** 13, n, dtype=I64)
        k[:4] = [-1, 0, -10 ** 15, O.I64_MIN + 5]
        sql["k"] = (SQL_DECIMAL, 2)
    elif kind == "char1":                                  # CHAR(1): bytes 0x01 .. 0xFF
        k = rng.integers(1, 256, n).astype(np.uint8)
        k[:255] = np.arange(1, 256, dtype=np.uint8)
    else:                                                  # BOOL
        k = rng.integers(0, 2, n).astype(np.uint8)
        sql["k"] = (SQL_BOOL, 0)
    if kind not in ("char1", "bool"):
        k[rng.integers(0, n, n // 4)] = k[rng.integers(0, n, n // 4)]
    k = rng.permutation(k)
    t = {"k": k, "id": _ids(n)}
    return OrderCase(name, t, ["k", "id"], [(0, asc)], sql=sql, path=path_of(n, -1))


# ---- digit structure of the radix keys -------------------------------------------------------------------------------
def digits(name, n, shape, asc):
    """BIGINT keys that differ only in some bits: every radix pass over a digit they agree in is skipped"""
    rng = _rng(name)
    base = I64(0x1234_5678_9ABC_DEF0 - 2 ** 63 + 2 ** 62)
    if shape == "equal":
        k, passes = np.full(n, base, I64), 0
    elif shape == "bit63":
        k, passes = np.where(rng.integers(0, 2, n) == 1, base ^ I64(O.I64_MIN), base).astype(I64), 1
    elif shape == "low":
        k, passes = (base & ~I64(0xF)) | rng.integers(0, 16, n, dtype=I64), 1
    else:                                                  # digit 9 (bits 36 .. 39)
        k, passes = (base & ~I64(0xF << 36)) | (rng.integers(0, 16, n, dtype=I64) << 36), 1
    t = {"k": k, "id": _ids(n)}
    return OrderCase(name, t, ["k", "id"], [(0, asc)], path="radix", passes=passes)


# ---- strings ------------------------------------------------------------------------------------------------------------
def str_values(rng, n, w):
    """n strings of at most w bytes: random ones (bytes 0x01 .. 0xFF), the empty string, 'AB' and 'AB ',
    groups that share a prefix of 7, 8, 9 or 16 bytes, and groups that differ only in the last byte at
    the declared width"""
    def rand(lo, hi):
        return bytes(rng.integers(1, 256, int(rng.integers(lo, hi + 1))).astype(np.uint8))
    pool = [b"", b"AB", b"AB ", b" ", b"A", b"\x80", b"\xff", b"B"]
    for p in (7, 8, 9, 16):
        pre = rand(min(p, w), min(p, w))
        pool += [pre + rand(0, w - len(pre)) for _ in range(6)] + [pre, pre[:-1] + b"\xff"]
    last = rand(w - 1, w - 1)
    pool += [last + bytes([b]) for b in (0x01, 0x20, 0x41, 0x7f, 0x80, 0xfe, 0xff)]
    pool = [s[:w] for s in pool]
    vals = [pool[i] for i in rng.integers(0, len(pool), n // 2)] + [rand(0, w) for _ in range(n - n // 2)]
    return np.array([vals[i] for i in rng.permutation(n)], dtype=f"S{w + 1}")


def strings(name, n, w, varchar, asc):
    rng = _rng(name)
    t = {"s": str_values(rng, n, w), "id": _ids(n)}
    sql = {"s": (SQL_VARCHAR, w)} if varchar else {}
    return OrderCase(name, t, ["id", "s"], [(1, asc)], sql=sql, path=path_of(n, -1))


def string_second(name, n):
    """a string key behind an INT key of few values: (INT ASC, VARCHAR(17) DESC, row id)"""
    rng = _rng(name)
    t = {"a": rng.integers(-3, 3, n).astype(np.int32), "s": str_values(rng, n, 17), "id": _ids(n)}
    return OrderCase(name, t, ["a", "s", "id"], [(0, True), (1, False)], sql={"s": (SQL_VARCHAR, 17)},
                     path=path_of(n, -1))


# ---- several keys ----------------------------------------------------------------------------------------------------------
def multi(name, n, keys, limit=-1):
    """every type, few values each, so that ties run through several keys; keys: [(column, ascending)]"""
    rng = _rng(name)
    t = {"b": rng.integers(-2, 2, n, dtype=I64) * (2 ** 62), "i": rng.integers(-3, 3, n).astype(np.int32),
         "c": rng.choice(np.array([0x01, 0x41, 0x80, 0xff], np.uint8), n), "f": rng.integers(0, 2, n).astype(np.uint8),
         "d": rng.integers(19920101, 19920104, n).astype(np.int32), "m": rng.integers(-2, 2, n, dtype=I64) * 100,
         "s8": np.array([b"ABCDEFGH", b"ABCDEFG", b"", b"\x80ABCDEFG"], "S9")[rng.integers(0, 4, n)],
         "v9": np.array([b"ABCDEFGH1", b"ABCDEFGH", b"ABCDEFGH\x81", b"AB "], "S10")[rng.integers(0, 4, n)],
         "id": _ids(n)}
    sql = {"f": (SQL_BOOL, 0), "d": (SQL_DATE, 0), "m": (SQL_DECIMAL, 2), "v9": (SQL_VARCHAR, 9)}
    out = list(t)
    return OrderCase(name, t, out, [(out.index(c), asc) for c, asc in keys], limit=limit, sql=sql, path=path_of(n, limit))


MULTI = {
    "keys2": [("i", True), ("b", False)],
    "keys3": [("c", False), ("v9", True), ("b", True)],
    "keys4": [("d", True), ("m", False), ("s8", False), ("f", True)],
    "keys5": [("f", False), ("i", True), ("s8", True), ("m", False), ("c", True)],
}
KEYS24 = [(c, j % 3 != 1) for j, c in zip(range(24), itertools.cycle(["i", "s8", "b", "c", "v9", "f", "d", "m"]))]


# ---- LIMIT and the radix select ----------------------------------------------------------------------------------------------
def limited(name, n, limit):
    """(k1 ASC, k2 DESC) with runs of about 80 equal k1 values, so that the second key decides at
    the cut, over a selection that keeps about 15 of 16 rows"""
    rng = _rng("limited")
    t = {"k1": rng.integers(-600, 600, n, dtype=I64), "k2": rng.integers(-50, 50, n).astype(np.int32),
         "f": rng.integers(0, 16, n).astype(np.uint8), "id": _ids(n)}
    kept = int((t["f"] > 0).sum())
    return OrderCase(name, t, ["k1", "k2", "id"], [(0, True), (1, False)], limit=limit, sel=("f", "GT", 0),
                     path=path_of(kept, limit))


def topk_case(name, t, out, order, limit, sql=None, fallback=False):
    """a case that takes the radix select at its GPU size (the bitonic sort at the oracle's)"""
    p = path_of(len(next(iter(t.values()))), limit)
    return OrderCase(name, t, out, order, limit=limit, sql=sql, path="topk->radix" if fallback and p == "topk" else p)


def tie_second_str(name, n):
    """k1 in runs of about 40; a VARCHAR second key decides at the cut"""
    rng = _rng(name)
    t = {"k1": rng.integers(0, n // 40, n, dtype=I64), "s": str_values(rng, n, 12), "id": _ids(n)}
    return topk_case(name, t, ["k1", "s", "id"], [(0, True), (1, True)], 1000, sql={"s": (SQL_VARCHAR, 12)})


def fallback_int(name, n):
    """5000 rows share the smallest first key: more candidates than one bitonic sort holds"""
    rng = _rng(name)
    k = rng.integers(0, 10 ** 9, n, dtype=I64)
    k[rng.choice(n, min(5000, n // 2), replace=False)] = -7
    t = {"k": k, "k2": rng.integers(0, 10 ** 6, n, dtype=I64), "id": _ids(n)}
    return topk_case(name, t, ["k", "k2", "id"], [(0, True), (1, False)], 10, fallback=True)


def _prefixed(rng, n, pre, share, w):
    """n CHAR(w) values; `share` of them start with the 8 bytes `pre` (the smallest first words)"""
    vals = [b"\x90" + bytes(rng.integers(1, 256, w - 1).astype(np.uint8)) for _ in range(n)]
    for i in rng.choice(n, min(share, n // 2), replace=False):
        vals[i] = pre + bytes(rng.integers(1, 256, int(rng.integers(0, w - 7))).astype(np.uint8))
    return np.array(vals, dtype=f"S{w + 1}")


def fallback_str(name, n):
    """a CHAR(20) first key; 5000 rows share their first 8 bytes, which only the radix sort tells apart"""
    rng = _rng(name)
    t = {"s": _prefixed(rng, n, b"AAAAAAAA", 5000, 20), "id": _ids(n)}
    return topk_case(name, t, ["s", "id"], [(0, True)], 100, fallback=True)


def topk_str(name, n):
    """a VARCHAR(16) first key, DESC; 3000 rows share their (largest) first 8 bytes"""
    rng = _rng(name)
    t = {"s": _prefixed(rng, n, b"\xff\xfe\xfd\xfc\xfb\xfa\xf9\xf8", 3000, 16), "id": _ids(n)}
    return topk_case(name, t, ["id", "s"], [(1, False)], 2048, sql={"s": (SQL_VARCHAR, 16)})


def bin_edge(name, n, lo, limit, asc=True):
    """unique keys lo, lo + 1, ... (permuted): the k-th is lo + limit - 1 ASC"""
    rng = _rng(name)
    t = {"k": lo + rng.permutation(n).astype(I64), "id": _ids(n)}
    return topk_case(name, t, ["k", "id"], [(0, asc)], limit)


def negative_first(name, n, asc):
    rng = _rng(name)
    k = -rng.integers(1, 10 ** 12, n, dtype=I64)
    k[rng.integers(0, n, n // 3)] = k[rng.integers(0, n, n // 3)]
    t = {"k": k, "x": rng.integers(-5, 5, n).astype(np.int32), "id": _ids(n)}
    return topk_case(name, t, ["k", "x", "id"], [(0, asc), (1, not asc)], 1500)


def extreme_kth(name, n, asc):
    """3 rows of INT64_MIN (ASC) or INT64_MAX (DESC) among random keys; LIMIT 2 cuts their tie"""
    rng = _rng(name)
    k = _wide(rng, n)
    k[rng.choice(n, 3, replace=False)] = O.I64_MIN if asc else O.I64_MAX
    t = {"k": k, "id": _ids(n)}
    return topk_case(name, t, ["k", "id"], [(0, asc)], 2)


def int32_desc(name, n):
    rng = _rng(name)
    k = rng.integers(O.I32_MIN, O.I32_MAX, n, dtype=I64, endpoint=True).astype(np.int32)
    k[:3] = [O.I32_MAX, O.I32_MAX, O.I32_MIN]
    t = {"k": rng.permutation(k), "id": _ids(n)}
    return topk_case(name, t, ["k", "id"], [(0, False)], 700)


# ---- sources of the final relation ------------------------------------------------------------------------------------------------
def grouped(name, n, groups, out, order, limit=-1):
    """GROUP BY g (BIGINT, negative too): g, SUM(v), COUNT(*), MIN(v), MAX(v), projected as `out`"""
    rng = _rng(name)
    t = {"g": rng.integers(0, groups, n, dtype=I64) * 7919 - 10 ** 6, "v": rng.integers(-10 ** 6, 10 ** 6, n, dtype=I64)}
    g = (["g"], [(AGG_SUM, "v"), (AGG_COUNT, None), (AGG_MIN, "v"), (AGG_MAX, "v")])
    return OrderCase(name, t, out, order, limit=limit, group=g, path=path_of(groups, limit))


def joined(name, n, limit):
    """t joins b on a unique key (one in 5 probe rows without a match): (id, x) of t, (y, s) of b"""
    rng = _rng(name)
    nb = n // 4
    b = {"bk": rng.permutation(nb).astype(I64) * 3, "y": rng.integers(-1000, 1000, nb, dtype=I64),
         "s": str_values(rng, nb, 9)}
    pk = rng.integers(0, nb, n, dtype=I64) * 3
    pk[::5] += 1
    t = {"pk": pk, "x": rng.integers(-9, 9, n).astype(np.int32), "id": _ids(n)}
    kept = n - len(pk[::5])
    return OrderCase(name, t, ["id", "x"], [(2, False), (3, True), (0, True)], limit=limit, join=(b, ["pk", "bk"], ["y", "s"]),
                     path=path_of(kept, limit))


# name: (builder of the case at n rows, n on the GPU, run interpreted too, takes the radix select on the GPU)
CASES = {}


def _add(name, fn, n, interp=False, topk=False):
    CASES[name] = (fn, n, interp, topk)


for _n in SIZES:
    _add(f"size_{_n}", lambda nm, n: sized(nm, n, passes=16 if n == 2_000_000 else None), _n, _n in (4096, 4097))
for _n in (4096, 4097, 100_003):
    _add(f"size_{_n}_desc", lambda nm, n: sized(nm, n, asc=False), _n)
for _kind in ("bigint", "int", "date", "decimal", "char1", "bool"):
    for _n in (3000, 50_000):
        for _asc in (True, False):
            _add(f"{_kind}_{_n}_{'asc' if _asc else 'desc'}", lambda nm, n, k=_kind, a=_asc: typed(nm, n, k, a), _n,
                 _kind == "bigint" and _n == 50_000)
for _shape in ("equal", "bit63", "low", "middle"):
    for _asc in (True, False):
        _add(f"digits_{_shape}_{'asc' if _asc else 'desc'}", lambda nm, n, s=_shape, a=_asc: digits(nm, n, s, a), 20_000,
             _shape == "bit63")
for _w in (2, 7, 8, 9, 15, 16, 17, 44):
    _add(f"char{_w}_asc", lambda nm, n, w=_w: strings(nm, n, w, False, True), 20_000, _w == 9)
    _add(f"varchar{_w}_desc", lambda nm, n, w=_w: strings(nm, n, w, True, False), 20_000)
for _w in (8, 9, 17):
    _add(f"char{_w}_desc_bitonic", lambda nm, n, w=_w: strings(nm, n, w, False, False), 4000)
    _add(f"varchar{_w}_asc_bitonic", lambda nm, n, w=_w: strings(nm, n, w, True, True), 4000)
_add("string_second", string_second, 30_000, True)
_add("string_second_bitonic", string_second, 2000)
for _k, _keys in MULTI.items():
    _add(f"{_k}_radix", lambda nm, n, ks=_keys: multi(nm, n, ks), 30_000, _k == "keys4")
    _add(f"{_k}_bitonic", lambda nm, n, ks=_keys: multi(nm, n, ks), 3000)
_add("keys24_radix", lambda nm, n: multi(nm, n, KEYS24), 20_000, True)
_add("keys24_bitonic", lambda nm, n: multi(nm, n, KEYS24), 4000)
_add("keys24_topk", lambda nm, n: multi(nm, n, KEYS24, 1000), 20_000, topk=True)
LIMITED_N = 100_003
for _lim in ("none", 0, 1, 2047, 2048, 2049, "n-1", "n", "n+1"):
    _add(f"limit_{_lim}", lambda nm, n, lim=_lim: limited(nm, n, {"none": -1, "n-1": n - 1, "n": n, "n+1": n + 1}.get(lim, lim)),
         LIMITED_N, _lim == 2048, _lim in (0, 1, 2047, 2048))
_add("limit_2048_bitonic", lambda nm, n: limited(nm, n, 2048), 4000)
_add("topk_tie_second_str", tie_second_str, 100_003, True, True)
_add("topk_fallback_int", fallback_int, 100_003, True, True)
_add("topk_fallback_str", fallback_str, 60_000, topk=True)
_add("topk_str_desc", topk_str, 60_000, topk=True)
_add("topk_kth_2047", lambda nm, n: bin_edge(nm, n, 0, 2048), 100_003, topk=True)
_add("topk_kth_2048", lambda nm, n: bin_edge(nm, n, 1, 2048), 100_003, topk=True)
_add("topk_kth_2pow22", lambda nm, n: bin_edge(nm, n, 2 ** 22 - 1000, 1001), 100_003, topk=True)
_add("topk_kth_2pow22_desc", lambda nm, n: bin_edge(nm, n, 2 ** 22 - n + 1000, 1000, False), 100_003, topk=True)
_add("topk_negative_asc", lambda nm, n: negative_first(nm, n, True), 100_003, topk=True)
_add("topk_negative_desc", lambda nm, n: negative_first(nm, n, False), 100_003, topk=True)
_add("topk_int64_min", lambda nm, n: extreme_kth(nm, n, True), 100_003, True, True)
_add("topk_int64_max_desc", lambda nm, n: extreme_kth(nm, n, False), 100_003, topk=True)
_add("topk_int32_desc", int32_desc, 100_003, topk=True)
_add("group_by_key_desc", lambda nm, n: grouped(nm, n, 30_000, [1, 0, 2], [(1, False)]), 200_000, True)
_add("group_by_sum_topk", lambda nm, n: grouped(nm, n, 30_000, [0, 1, 2, 3, 4], [(1, False), (0, True)], 100), 200_000,
     topk=True)
_add("group_by_count_bitonic", lambda nm, n: grouped(nm, n, 1000, [2, 0, 3, 4], [(0, False), (1, True)]), 200_000)
_add("join_late_topk", lambda nm, n: joined(nm, n, 2047), 200_000, True, True)
_add("join_late_radix", lambda nm, n: joined(nm, n, -1), 200_000)
SMALL = 3000          # rows of the instances the oracle checks


def make(name, n=None):
    fn, big, _, _ = CASES[name]
    return fn(name, big if n is None else min(n, big))


def uses_topk(c):
    return c.path in ("topk", "topk->radix")


def expected_candidates(c, want):
    """the rows a radix select keeps: first-key value (the first 8 bytes of a string) not beyond the
    k-th one's"""
    col, asc = want[c.order[0][0]], c.order[0][1]
    if col.dtype == object:
        col = np.array([s[:8].ljust(8, b"\0") for s in col], dtype=object)
    kth = col[max(c.limit, 1) - 1]
    return int(sum(1 for x in col if (x <= kth if asc else x >= kth)))


# ---- GPU ----------------------------------------------------------------------------------------------------------
OPTIONS = {"topk": 1, "specialize": 1, "late_materialize": 1, "trace": 0}


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


@lru_cache(maxsize=2)
def case_and_want(name):
    c = make(name)
    return c, O.reference(c)


_TAGS = itertools.count(1)
ORDER_LINE = re.compile(r"\[rq\] order by: n=(\d+) path=(\S+)(?: candidates=(\d+))?(?: passes=(\d+))?")


def check_path(c, want, err, topk):
    """the careful execution's trace names the path case c declares"""
    assert re.search(r"careful run rc=0", err), f"{c.name}: no trace of a careful execution"
    lines = ORDER_LINE.findall(err)
    path = "radix" if not topk and uses_topk(c) else c.path
    n = len(want[0])
    if path == "none":
        assert not lines, f"{c.name}: sorted {lines}"
        return
    assert len(lines) == 1, f"{c.name}: {len(lines)} order by lines: {lines}"
    got_n, got_path, cand, passes = lines[0]
    what = f"{c.name} (topk={topk}): {lines[0]}"
    assert int(got_n) == n and got_path == path, what
    if path.startswith("topk"):
        assert int(cand) == expected_candidates(c, want), what
    if path.endswith("radix") and c.passes is not None:
        assert int(passes) == c.passes, what


def upload(engine, c):
    return {name: engine.upload(name, cols) for name, cols in c.tables().items()}


def execute_five_times(engine, capfd, c, want, topk=1, spec=1, handles=None, tag=None):
    """runs case c: careful (traced), replayed, captured, graph, graph; every result must be one the
    reference allows. Returns the first execution's trace."""
    from resql_b200 import Plan
    sql = O.result_sql(c)
    plan = Plan(O.order_plan(c, next(_TAGS) if tag is None else tag))
    own = handles is None
    h = upload(engine, c) if own else handles
    try:
        engine.set_option("topk", topk)
        engine.set_option("specialize", spec)
        engine.set_option("late_materialize", 2 if c.join else 1)
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
    what = f"{c.name} topk={topk} specialize={spec}"
    for run, res in enumerate(results):
        O.assert_ordered_equal(res.columns, want, sql, c.order, c.limit, f"{what} execution {run + 1}")
    return err


GPU_RUNS = [run for name, (_, _, interp, topk) in CASES.items()
            for run in [(name, 1, 1)] + [(name, 0, 1)] * topk + [(name, 1, 0)] * interp]


@pytest.mark.parametrize("name,topk,spec", GPU_RUNS, ids=[f"{n}-topk{t}-spec{s}" for n, t, s in GPU_RUNS])
def test_order_by(name, topk, spec, engine, capfd):
    c, want = case_and_want(name)
    err = execute_five_times(engine, capfd, c, want, topk, spec)
    check_path(c, want, err, topk)


def test_more_than_24_keys_are_refused(engine):
    from resql_b200 import EngineError, Plan
    c = multi("keys25", 5000, KEYS24 + [("id", True)])
    h = upload(engine, c)
    try:
        with pytest.raises(EngineError) as e:
            engine.execute(Plan(O.order_plan(c)), h)
        assert e.value.code == RQ_ERR_UNSUPPORTED
        c.order = [(len(c.out), True)]
        with pytest.raises(EngineError) as e:
            engine.execute(Plan(O.order_plan(c)), h)
        assert e.value.code == RQ_ERR_INVALID
    finally:
        for t in h.values():
            t.free()


# ---- changed data under a recorded plan ---------------------------------------------------------------------------
def _radix_digits(n, changed):
    """keys 0 .. 0xF00 that vary in digit 2 only, then in every digit up to it (the same min and max)"""
    rng = _rng("changed_radix")
    k = rng.integers(0, 16, n, dtype=I64) << 8 if not changed else rng.integers(0, 0xF00, n, dtype=I64, endpoint=True)
    k[:2] = [0, 0xF00]
    return k, "radix"


def _kth_moves(n, changed):
    rng = _rng("changed_kth" + str(changed))
    k = rng.integers(0, 10 ** 6, n, dtype=I64)
    k[:2] = [0, 10 ** 6]
    return k, "topk"


def _to_fallback(n, changed):
    """the 6000 smallest keys all equal (more candidates than one bitonic sort holds), or distinct"""
    rng = _rng("changed_fallback")
    k = rng.integers(1000, 10 ** 6, n, dtype=I64)
    k[2:6002] = 1 if changed else np.arange(1, 6001)
    k[:2] = [0, 10 ** 6]
    return k, ("topk->radix" if changed else "topk")


def _from_fallback(n, changed):
    k, path = _to_fallback(n, not changed)
    return k, path


CHANGES = {"radix_digit_varies": (_radix_digits, -1), "topk_kth_moves": (_kth_moves, 100),
           "topk_to_fallback": (_to_fallback, 50), "fallback_to_topk": (_from_fallback, 50)}


@pytest.mark.parametrize("change", sorted(CHANGES))
def test_changed_borrowed_data_under_a_recorded_plan(change, engine, capfd):
    """one plan over a borrowed table: five executions (the last two from the graph), then the same
    memory holds other keys (the same minimum and maximum, so the table's upload statistics still
    hold) and the plan runs five times more. A prediction the new keys make wrong (a varying-bits
    mask, a candidate count) is noticed on the device and the plan reruns the careful way."""
    import torch
    from resql_b200.native import RQ_I64
    gen, limit = CHANGES[change]
    n = 50_000
    dev = {"k": torch.from_numpy(gen(n, False)[0]).cuda(), "id": torch.from_numpy(_ids(n)).cuda()}
    torch.cuda.synchronize()
    h = {"t": engine.upload_device("t", {c: (x.data_ptr(), RQ_I64, 8) for c, x in dev.items()}, n)}
    tag = next(_TAGS)
    try:
        for changed in (False, True):
            k, path = gen(n, changed)
            dev["k"].copy_(torch.from_numpy(k))
            torch.cuda.synchronize()
            c = OrderCase(f"{change}_{int(changed)}", {"k": k, "id": _ids(n)}, ["k", "id"], [(0, True)], limit=limit,
                          path=path)
            want = O.reference(c)
            err = execute_five_times(engine, capfd, c, want, handles=h, tag=tag)
            if changed and change == "topk_kth_moves":
                # the candidate count is the same, so no prediction is wrong: the graph selects the new
                # k-th value on the device, and its result (checked above) stands
                assert "careful run" not in err, f"{change}: the graph's result was discarded\n{err[-2000:]}"
                continue
            if changed:
                assert "graph result discarded" in err, f"{change}: the stale prediction went unnoticed\n{err[-2000:]}"
            check_path(c, want, err, 1)
    finally:
        h["t"].free()
        torch.cuda.synchronize()
