"""Python model of a materialize lowered in sink rounds (engine_exec.inl "sink rounds"), on top of
tests/vm_model.py: the host-level units printed by rq_debug_lower run in order over whole numpy columns,
and every round's values are read from their slots right after the round's last unit, as the round
variant of the scan kernel stores them. A value read after its slot was reused by a later round, or a
round whose units drop tuples, shows up as a difference from the plan oracle.
Test infrastructure only."""
import numpy as np

from oracle import plan_oracle as PO
from resql_b200 import native as N
import vm_model as V


def parse_rounds(text):
    """(prefix end, [(unit begin, unit end, value begin, value end)]); None without rounds"""
    prefix, rounds = None, []
    for line in text.splitlines():
        f = line.split()
        if f[0] == "rounds":
            prefix = int(f[3])
        elif f[0] == "round":
            rounds.append((int(f[3]), int(f[4]), int(f[6]), int(f[7])))
    return None if prefix is None else (prefix, rounds)


def lower_text(plan, pi, src_cols, with_stats=True):
    types, widths, mins, maxs = [], [], [], []
    for a in src_cols:
        t, w = V.phys_of(a)
        types.append(t); widths.append(w)
        if with_stats and a.dtype.kind in "iu" and len(a):
            mins.append(int(a.min())); maxs.append(int(a.max()))
        else:
            mins.append(1); maxs.append(0)
    return N.debug_lower(plan, pi, V.IMPL_EMIT, types, widths, mins, maxs)


def run_rounds_vm(plan, pi, src_cols, with_stats=True):
    """Output columns of a materialize pipeline over a table's columns, through its round schedule."""
    text = lower_text(plan, pi, src_cols, with_stats)
    prog = V.parse(text)
    sched = parse_rounds(text)
    assert sched is not None, "the pipeline was not lowered in rounds"
    prefix, rounds = sched
    vals = [PO._to_value(a) for a in src_cols]
    n = len(vals[0]) if vals else 0
    valid = np.ones(n, dtype=bool)
    slots = {}

    def operand(kind, idx, imm):
        if kind == V.S_COL:
            return vals[prog["cols"][idx]]
        if kind == V.S_STR:
            return vals[prog["strcols"][idx]]
        if kind == V.S_SLOT:
            return slots[idx]
        if kind == V.S_IMM:
            return np.full(n, imm, dtype=np.int64)
        return None

    def vref(kind, idx):
        return operand(V.S_IMM, 0, prog["imm"][idx]) if kind == V.S_IMM else operand(kind, idx, 0)

    outs = [None] * len(prog["out"])

    def store(u):           # the rounds whose units end at u store their values now
        for ub, ue, vb, ve in rounds:
            if ue == u and u >= prefix:
                for v in range(vb, ve):
                    outs[v] = vref(*prog["out"][v]).copy()

    old = np.seterr(over="ignore")
    units = prog["unit"]
    store(0)
    for u, (op, gop, xk, xi, ximm, yk, yi, yimm, zk, zi, zimm, imm, dst, filt, aux, imm2, n32) in enumerate(units):
        x, y, z = operand(xk, xi, ximm), operand(yk, yi, yimm), operand(zk, zi, zimm)
        if u >= prefix:
            assert op not in (V.H_FCMP, V.H_FRANGE, V.H_PROBE) and not filt, "a unit after the prefix drops tuples"
        if op == V.H_FCMP:
            valid = valid & (V._binop(gop, x, np.full(n, imm, dtype=np.int64), valid) != 0)
        elif op == V.H_FRANGE:
            valid = valid & np.array([imm <= v <= imm + (imm2 & 0xFFFFFFFFFFFFFFFF) for v in x.astype(object)], dtype=bool)
        else:
            if op == V.H_BIN:
                t = V._binop(gop, x, y, valid)
                if n32 and gop == V.D_MUL:
                    t = ((x.astype(np.uint64) & np.uint64(0xFFFFFFFF)) * (y.astype(np.uint64) & np.uint64(0xFFFFFFFF))).astype(np.int64)
            elif op == V.H_MULI:
                inner = V._binop(gop, x, np.full(n, imm, dtype=np.int64), valid)
                t = ((inner.astype(np.uint64) & np.uint64(0xFFFFFFFF)) * (y.astype(np.uint64) & np.uint64(0xFFFFFFFF))).astype(np.int64) if n32 else inner * y
            elif op == V.H_SEL:
                t = np.where((x & 0xFF) != 0, y, z)
            else:
                raise NotImplementedError(op)
            if dst >= 0:
                slots[dst] = t
            if filt:
                valid = valid & ((t & 0xFF) != 0)
        store(u + 1)
    np.seterr(**old)
    assert all(o is not None for o in outs)
    return [o[valid] for o in outs]
