"""Sink rounds without a GPU: rq_debug_lower prints the round schedule of a materialize whose computed
outputs need more than the 12 value slots (the prefix's units, then each round's units and values),
and tests/vm_model_rounds.py runs the printed program round by round against the plan oracle. Plans
that fit the single sink lower exactly as before under the default option."""
import contextlib

import numpy as np
import pytest

from oracle.plan_oracle import run_plan
from resql_b200 import EngineError, Plan
from resql_b200 import native as N
import vm_model_rounds as VR
from test_gpu_sink_rounds import computed_select, random_wide_plan, table

RQ_ERR_UNSUPPORTED = 3


@contextlib.contextmanager
def sink_rounds(v):
    lib = N.load()
    lib.rq_set_option(b"sink_rounds", float(v))
    try:
        yield
    finally:
        lib.rq_set_option(b"sink_rounds", 1.0)


def src(tabs):
    return [tabs["t"][c] for c in ("k", "v", "d")]


def lower(d, tabs):
    return VR.lower_text(Plan(d), 0, src(tabs))


def agrees_with_oracle(d, tabs):
    got = VR.run_rounds_vm(Plan(d), 0, src(tabs))
    want = run_plan(d, tabs)[0]
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert np.array_equal(np.asarray(g, dtype=np.int64), np.asarray(w, dtype=np.int64))


def schedule(text):
    sched = VR.parse_rounds(text)
    slots = int(next(l.split()[5] for l in text.splitlines() if l.startswith("cols ")))
    return sched, slots


def test_twelve_computed_outputs_fit_one_sink():
    tabs = table(100, seed=1)
    sched, slots = schedule(lower(computed_select(12, filt=500), tabs))
    assert sched is None and slots == 12


@pytest.mark.parametrize("m,n_rounds", [(13, 2), (24, 2), (64, 6)])
@pytest.mark.parametrize("shared", [False, True])
def test_wide_computed_select_lowers_in_rounds(m, n_rounds, shared):
    tabs = table(3000, seed=m)
    text = lower(computed_select(m, shared=shared, filt=500), tabs)
    (prefix, rounds), slots = schedule(text)
    assert slots <= 12
    # values in order, every round non-empty, units contiguous behind the prefix
    assert rounds[0][2] == 0 and rounds[-1][3] == m
    assert all(r[2] < r[3] for r in rounds)
    assert all(a[3] == b[2] and a[1] == b[0] for a, b in zip(rounds, rounds[1:]))
    assert rounds[0][0] == prefix
    if not shared:
        assert len(rounds) == n_rounds
    agrees_with_oracle(computed_select(m, shared=shared, filt=500), tabs)


def test_the_prefix_holds_the_filter_and_nothing_after_it_drops_tuples():
    tabs = table(2000, seed=3)
    d = computed_select(30, filt=200)
    prefix, rounds = VR.parse_rounds(lower(d, tabs))
    assert prefix >= 1
    agrees_with_oracle(d, tabs)      # (the model asserts that no unit after the prefix filters)


@pytest.mark.parametrize("m", [1, 5, 10])
def test_forced_rounds_on_plans_that_fit(m):
    tabs = table(1000, seed=m)
    d = computed_select(m, shared=True, filt=600)
    assert VR.parse_rounds(lower(d, tabs)) is None
    with sink_rounds(2):
        assert VR.parse_rounds(lower(d, tabs)) is not None
        agrees_with_oracle(d, tabs)


@pytest.mark.parametrize("seed", range(10))
def test_plans_that_fit_lower_as_before(seed):
    """the default option changes nothing where the single sink holds the values"""
    tabs = table(500, seed=seed)
    d = computed_select(2 + seed, shared=seed % 2 == 1, filt=300)
    with sink_rounds(0):
        before = lower(d, tabs)
    assert lower(d, tabs) == before


@pytest.mark.parametrize("seed", range(60))
def test_random_wide_plans_agree_with_the_oracle(seed):
    tabs = table(int(np.random.default_rng(seed).integers(1, 3000)), seed=1000 + seed)
    agrees_with_oracle(random_wide_plan(seed), tabs)


def test_65_outputs_are_refused():
    tabs = table(10, seed=0)
    with pytest.raises(EngineError) as e:
        lower(computed_select(65), tabs)
    assert e.value.code == RQ_ERR_UNSUPPORTED


def test_rounds_off_keeps_the_refusal():
    tabs = table(10, seed=0)
    with sink_rounds(0), pytest.raises(EngineError) as e:
        lower(computed_select(13), tabs)
    assert e.value.code == RQ_ERR_UNSUPPORTED
