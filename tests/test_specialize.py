"""Run-time specialization of the scan kernel (csrc/jit.h).

CPU: the specialization of every golden plan's scan pipelines (probing ones against placeholder build
sides) compiles with NVRTC for sm_100a; the kernels of Q1, Q6 and Q3's orders and lineitem pipelines fit
128 registers without spills or a stack frame; the program baked into the generated source is the one
rq_debug_lower prints.
GPU: golden, fuzzed and aggregation-limit plans give identical results with specialization off and on,
every plan launches specialized kernels with it on, and a replayed plan's CUDA graph holds them."""
import re

import numpy as np
import pytest

from common import plan_names, load_plan_dict, plan_tables, serialize_columns
from resql_b200 import native as N
from resql_b200.plan import Plan, OP
import vm_model

IMPL_GROUPJOIN = 6


def _meta(d, pi, tables):
    t = d["tables"][d["pipelines"][pi]["source_id"]]
    types, widths, mn, mx = [], [], [], []
    for c in t["columns"]:
        a = np.asarray(tables[t["name"]][c])
        if a.dtype == object:
            types.append(N.RQ_STR)
            widths.append(max((len(x) for x in a), default=1) + 1)
        else:
            ty, w = vm_model.phys_of(a)
            types.append(ty)
            widths.append(w)
        if a.dtype.kind in "iu" and len(a):
            mn.append(int(a.min())); mx.append(int(a.max()))
        else:
            mn.append(1); mx.append(0)
    return types, widths, mn, mx


def _impl(d, pi):
    """the sink implementation the executor picks first for pipeline pi"""
    p = d["pipelines"][pi]
    if p["sink_kind"] == 2:
        return vm_model.IMPL_BUILD
    if p["sink_kind"] == 3:
        return vm_model.IMPL_EMIT
    if not any(n[0] == OP["PROBE"] for n in p["nodes"]):
        return vm_model.IMPL_REGAGG
    gj = int(N.debug_lower(Plan(d), pi, IMPL_GROUPJOIN, [], []).split()[1])
    return IMPL_GROUPJOIN if gj >= 0 else vm_model.IMPL_HASHAGG


def _scan_pipelines(d):
    return [pi for pi, p in enumerate(d["pipelines"]) if p["source_kind"] == 1]


def _specialize(name, sf001):
    d = load_plan_dict(name)
    tables = plan_tables(d, sf001)
    out = []
    for pi in _scan_pipelines(d):
        impl = _impl(d, pi)
        try:
            text = N.debug_specialize(Plan(d), pi, impl, *_meta(d, pi, tables))
        except N.EngineError as e:
            if "does not lower" in str(e) or "unsupported" in str(e).lower():
                continue
            raise
        out.append((d, pi, impl, text))
    return out


def _kernel_resources(text):
    log = text.split("---- log ----")[1]
    m = re.search(r"Function properties for _ZN2rq14rq_scan_kernel\w*\s*\n\s*ptxas\s*\.\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                  r"(\d+) bytes spill loads\s*\n\s*ptxas info\s*: Used (\d+) registers", log)
    assert m, log
    stack, st, ld, regs = (int(x) for x in m.groups())
    return regs, stack, st + ld


@pytest.mark.parametrize("name", plan_names())
def test_specialization_compiles(name, sf001):
    for d, pi, impl, text in _specialize(name, sf001):
        assert text.rstrip().endswith("status ok"), text.split("---- log ----")[1]


@pytest.mark.parametrize("name,pipelines", [("q1", [0]), ("q6", [0]), ("q3", [1, 2])])
def test_bench_kernels_fit(name, pipelines, sf001):
    """the bench's scans: Q1, Q6, and Q3's orders (probe customer, build) and lineitem (probe orders,
    groupjoin) pipelines"""
    got = {pi: _kernel_resources(text) for d, pi, impl, text in _specialize(name, sf001)}
    for pi in pipelines:
        regs, stack, spills = got[pi]
        assert regs <= 128 and stack == 0 and spills == 0, (name, pi, regs, stack, spills)


@pytest.mark.parametrize("name", ["q1", "q6", "q3", "sel_or", "case_sum", "sel_strings"])
def test_baked_program_is_the_lowered_one(name, sf001):
    for d, pi, impl, text in _specialize(name, sf001):
        if any(n[0] == OP["PROBE"] for n in d["pipelines"][pi]["nodes"]):
            continue        # (rq_debug_lower has no build sides to probe)
        baked = [tuple(int(x) for x in m) for m in
                 re.findall(r"case \d+: u = UInsn\{(\d+), (\d+), (\d+), (\d+), (\d+), (\d+), (\d+), 0, (\d+)u, (\d+)u, 0, (\d+)u, (\d+)u\}", text)]
        lowered = []
        tables = plan_tables(d, sf001)
        for line in N.debug_lower(Plan(d), pi, impl, *_meta(d, pi, tables)).splitlines():
            f = line.split()
            if f[0] == "uinsn":
                code, flags, dst, aux, gop, xk, yk, zk, xr, yr, zr = (int(x) for x in f[1:12])
                lowered.append((code, flags, gop, aux, xk, yk, zk, xr, dst, yr, zr))
        assert baked == lowered


# ---- GPU: the same results with and without specialization ---------------------------------------------
def _run(eng, d, tabs, specialize):
    N.load().rq_set_option(b"specialize", float(specialize))
    try:
        handles = {n: eng.upload(n, c) for n, c in tabs.items()}
        res, _ = eng.execute(Plan(d), handles)
        rows = sorted(serialize_columns(res.columns, res.sql_types, res.sql_widths))
        for h in handles.values():
            h.free()
        return rows
    finally:
        N.load().rq_set_option(b"specialize", 1.0)


def _agg_limit_cases():
    """aggregation plans of tests/agg_limit_plans.py over a table t(k, v, w): grouped and ungrouped
    sums near the 32-bit accumulator forms, and a computed value"""
    import agg_limit_plans as A
    rng = np.random.default_rng(3)
    n = 300_000
    t = {"t": {"k": rng.integers(0, 4, n).astype(np.int64), "v": rng.integers(0, 1 << 31, n).astype(np.int64),
               "w": rng.integers(-(1 << 40), 1 << 40, n).astype(np.int64)}}
    return [("agg_limit_sum_by_k", A.sum_by(["k", "v", "w"], ["k"], "v"), t),
            ("agg_limit_sum", A.sum_by(["k", "v", "w"], [], "v"), t),
            ("agg_limit_sub", A.sum_by(["k", "v", "w"], ["k"], lambda p: p.n("SUB", p.col("v"), p.col("w"))), t)]


def _cases(data):
    import plan_fuzz
    out = [(n, load_plan_dict(n)) for n in plan_names()] + [(f"fuzz_{s}", plan_fuzz.random_plan(s)) for s in range(8)]
    return [(n, d, plan_tables(d, data)) for n, d in out] + _agg_limit_cases()


@pytest.mark.gpu
def test_specialized_results_identical(sf001):
    from resql_b200 import Engine
    eng = Engine(0)
    for name, d, tabs in _cases(sf001):
        before = N.specialized_launches()
        generic = _run(eng, d, tabs, 0)
        assert N.specialized_launches() == before, f"{name}: specialize=0 launched specialized kernels"
        spec = _run(eng, d, tabs, 1)
        assert spec == generic, name
        assert N.specialized_launches() > before, f"{name}: no launch ran a specialized kernel"


@pytest.mark.gpu
def test_replayed_graph_holds_specialized_kernels(sf001):
    """a plan executed repeatedly is replayed and then captured into a CUDA graph (engine_exec.inl
    "host reads of device values"): the capture records the cached specializations"""
    from resql_b200 import Engine
    eng = Engine(0)
    d = load_plan_dict("q6")
    tabs = plan_tables(d, sf001)
    handles = {n: eng.upload(n, c) for n, c in tabs.items()}
    before = N.specialized_launches(captured=True)
    rows = []
    for _ in range(4):
        res, _ = eng.execute(Plan(d), handles)
        rows.append(sorted(serialize_columns(res.columns, res.sql_types, res.sql_widths)))
    for h in handles.values():
        h.free()
    assert all(r == rows[0] for r in rows)
    assert N.specialized_launches(captured=True) > before
