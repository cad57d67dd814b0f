"""CPU checks of the ORDER BY test infrastructure (order_plans.py): the reference agrees with the plan
oracle on small instances of every case of test_gpu_order_by.py, each case declares the sort path its
GPU size takes, and the tie-aware comparison rejects wrong results that a comparison of key sequences
and tuple multisets alone would let through."""
import numpy as np
import pytest

import order_plans as O
from oracle.plan_oracle import run_plan
from test_gpu_order_by import CASES, SMALL, BITONIC_MAX, make, path_of, expected_candidates, uses_topk


@pytest.mark.parametrize("name", sorted(CASES))
def test_reference_matches_the_oracle(name):
    c = make(name, SMALL)
    d = O.order_plan(c)
    got, st, sw = run_plan(d, c.tables())
    sql = O.result_sql(c)
    assert [tuple(x) for x in zip(st, sw)] == sql, name
    O.assert_ordered_equal(got, O.reference(c), sql, c.order, c.limit, f"{name} (oracle)")


def radix_passes(c, want):
    """the digit passes of the engine's radix sort: 4-bit digits that vary over the order-preserving
    64-bit keys of each key word (sign bit flipped, complemented for DESC; strings in 8-byte words)"""
    passes = 0
    for i, asc in c.order:
        col, (t, w) = want[i], O.result_sql(c)[i]
        if col.dtype == object:
            pad = np.array([s.ljust((w + 7) // 8 * 8, b"\0") for s in col], dtype=object)
            words = [np.array([int.from_bytes(s[8 * j:8 * j + 8], "big") for s in pad], np.uint64) for j in range((w + 7) // 8)]
        else:
            words = [col.astype(np.int64).view(np.uint64) ^ np.uint64(2 ** 63)]
        for k in words:
            k = k if asc else ~k
            varying = int(np.bitwise_or.reduce(k)) ^ int(np.bitwise_and.reduce(k))
            passes += sum(1 for s in range(0, 64, 4) if (varying >> s) & 15)
    return passes


@pytest.mark.parametrize("name", sorted(CASES))
def test_cases_declare_their_path(name):
    """at its GPU size: the path the case declares is the one its row count, LIMIT and candidate count
    select, and the radix passes it declares are the digits its keys vary in"""
    c = make(name)
    want = O.reference(c)
    n = len(want[0])
    path = path_of(n, c.limit)
    if path == "topk" and expected_candidates(c, want) > BITONIC_MAX:
        path = "topk->radix"
    assert c.path == path, f"{name}: declares {c.path}, takes {path} ({n} rows, LIMIT {c.limit})"
    assert CASES[name][3] == uses_topk(c), name
    if c.passes is not None:
        assert radix_passes(c, want) == c.passes, name


def test_the_matrix_covers_every_path():
    paths = {make(name).path for name in CASES if CASES[name][1] <= 10 ** 5}
    assert paths >= {"none", "bitonic", "radix", "topk", "topk->radix"}
    assert {0, 16} <= {make(name).passes for name in CASES if name.startswith(("digits_", "size_2000000"))}


# ---- the comparison itself -----------------------------------------------------------------------------------------------
SQL = [(O.SQL_BIGINT, 0), (O.SQL_VARCHAR, 4)]
ORDER = [(0, True)]


def _cols(rows):
    return [np.array([r[0] for r in rows], np.int64), np.array([r[1] for r in rows], "S5")]


WANT = _cols([(1, b"a"), (1, b"b"), (2, b"c"), (2, b"d"), (2, b"e"), (3, b"f")])


def check(rows, limit=-1):
    O.assert_ordered_equal(_cols(rows), WANT, SQL, ORDER, limit, "hand-made")


def test_accepts_any_order_inside_ties():
    check([(1, b"b"), (1, b"a"), (2, b"e"), (2, b"c"), (2, b"d"), (3, b"f")])
    check([(1, b"a"), (1, b"b"), (2, b"e")], limit=3)
    check([(1, b"b"), (1, b"a"), (2, b"d"), (2, b"c")], limit=4)


def test_rejects_a_wrong_row_inside_a_tie_run():
    with pytest.raises(AssertionError, match="inside a run"):
        check([(1, b"a"), (1, b"a"), (2, b"c"), (2, b"d"), (2, b"e"), (3, b"f")])


def test_rejects_a_row_from_outside_the_cut_tie_group():
    with pytest.raises(AssertionError, match="LIMIT cuts"):
        check([(1, b"a"), (1, b"b"), (2, b"f")], limit=3)
    with pytest.raises(AssertionError, match="LIMIT cuts"):
        check([(1, b"a"), (1, b"b"), (2, b"c"), (2, b"c")], limit=4)


def test_rejects_a_swapped_order():
    with pytest.raises(AssertionError, match="key sequence"):
        check([(1, b"a"), (2, b"c"), (1, b"b"), (2, b"d"), (2, b"e"), (3, b"f")])
    with pytest.raises(AssertionError, match="key sequence"):
        check([(1, b"a"), (1, b"b"), (3, b"f")], limit=3)


def test_rejects_a_wrong_row_count():
    with pytest.raises(AssertionError, match="rows"):
        check([(1, b"a"), (1, b"b")], limit=3)


def test_descending_strings_compare_unsigned_with_trailing_blanks():
    """the reference orders strings as strcmp does: unsigned bytes, a prefix first, blanks count"""
    t = {"s": np.array([b"AB ", b"\x80", b"AB", b"", b"A\xff", b"AB!"], "S4")}
    c = O.OrderCase("strcmp", t, ["s"], [(0, False)], sql={"s": (O.SQL_VARCHAR, 3)})
    assert list(O.reference(c)[0]) == [b"\x80", b"A\xff", b"AB!", b"AB ", b"AB", b""]
