"""CPU-only check of the groupjoin decision (engine_exec.inl groupjoin_probe): which aggregation
pipelines group by the key of a join whose build has no other consumer, so that they aggregate into
the entries of a direct-address build instead of a hash table of their own."""
import copy

import pytest

from common import plan_names, load_plan_dict
from resql_b200 import native as N
from resql_b200.plan import Plan

IMPL_GROUPJOIN = 6


def _decision(d, pi):
    out = N.debug_lower(Plan(d), pi, IMPL_GROUPJOIN, [], [])
    f = out.split()
    assert f[0] == "groupjoin"
    return int(f[1])


# fixture -> {aggregation pipeline: PROBE node of its (simplified) program}
QUALIFY = {"q3": {2: 7}}


@pytest.mark.parametrize("name", plan_names())
def test_which_fixture_pipelines_qualify(name):
    d = load_plan_dict(name)
    got = {pi: _decision(d, pi) for pi, p in enumerate(d["pipelines"]) if p["sink_kind"] == 1}
    want = {pi: QUALIFY.get(name, {}).get(pi, -1) for pi in got}
    assert got == want


def _q3_with_keys(nodes):
    d = copy.deepcopy(load_plan_dict("q3"))
    p = d["pipelines"][2]
    p["keys"] = [[n, 0, 3, 0] for n in nodes]
    return d


def test_q3_key_sets():
    # nodes of Q3's lineitem pipeline: 0 l_orderkey, 7 PROBE orders, 8 PAYLOAD o_orderkey (repeats the
    # build key), 9 PAYLOAD o_orderdate, 10 PAYLOAD o_shippriority, 15 revenue
    assert _decision(_q3_with_keys([0, 9, 10]), 2) == 7
    assert _decision(_q3_with_keys([8, 9, 10]), 2) == 7        # the join key's repeat instead of the column
    assert _decision(_q3_with_keys([9, 8]), 2) == 7
    assert _decision(_q3_with_keys([9, 10]), 2) == -1          # groups are not one per entry
    assert _decision(_q3_with_keys([0, 1]), 2) == -1           # a key that is not an attribute of the joined row
    assert _decision(_q3_with_keys([15]), 2) == -1


def test_q3_not_with_a_second_consumer_or_a_string_key():
    d = copy.deepcopy(load_plan_dict("q3"))
    # a second pipeline probing the orders build: the entries cannot hold two consumers' groups
    second = copy.deepcopy(d["pipelines"][2])
    second["sink_kind"] = 3
    second["keys"] = []
    second["vals"] = [[0, 0, 3, 0]]
    d["pipelines"].insert(3, second)
    assert _decision(d, 2) == -1
    d = _q3_with_keys([0, 9])
    d["pipelines"][2]["keys"][1] = [9, 0, 1, 15]               # CHAR(15): string keys keep the hash path
    assert _decision(d, 2) == -1
