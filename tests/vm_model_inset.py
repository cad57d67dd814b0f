"""The Python models of the VM (tests/vm_model.py) with the IN-list set test added: the host unit H_INSET
and the generic device unit's operation D_INSET, t = (x in the constant set at imm). rq_debug_lower prints
each set decoded from its device form (`inset <address> <form> <n>`, then one `insetv <address> <member>`
per member: integers, or hex bytes of a string constant, '-' for the empty string).

The models are run unchanged: an H_INSET unit is handed to the host model as the equivalent H_BIN unit
with operation D_INSET and the set's address as its constant operand, and the models' binary-operation
evaluator is given D_INSET, for the duration of one run only. Test infrastructure only."""
import contextlib

import numpy as np

import vm_model as _VM
from vm_model import *  # noqa: F401,F403  (constants and helpers of the base models)
from resql_b200 import native as _N

H_INSET = 7                                      # engine.cu HOp
D_INSET = 23                                     # rq_internal.h DOp
IS_BITMAP, IS_SORTED, IS_CHAR, IS_VARCHAR = range(4)     # rq_internal.h InSetForm


def parse_sets(text):
    """device address -> (form, members); integers as ints, string constants as bytes"""
    sets = {}
    for line in text.strip().split("\n"):
        f = line.split()
        if f[0] == "inset":
            sets[int(f[1])] = (int(f[2]), set())
        elif f[0] == "insetv":
            form, mem = sets[int(f[1])]
            mem.add(int(f[2]) if form in (IS_BITMAP, IS_SORTED) else (b"" if f[2] == "-" else bytes.fromhex(f[2])))
    return sets


def in_set(sets, addr, x, valid):
    """1 where x is in the set (CHAR sets compare without trailing blanks); strings of tuples outside
    `valid` are not looked at, like on the device"""
    form, mem = sets[addr]
    if form in (IS_BITMAP, IS_SORTED):
        return np.isin(np.asarray(x).astype(np.int64), np.array(sorted(mem), dtype=np.int64)).astype(np.int64)
    norm = (lambda u: u.rstrip(b" ")) if form == IS_CHAR else (lambda u: u)
    return np.array([1 if ok and norm(u) in mem else 0 for u, ok in zip(x, valid)], dtype=np.int64)


def parse(text):
    """vm_model.parse plus the sets (`sets`); H_INSET units stay as printed"""
    prog = _VM.parse(text)
    prog["sets"] = parse_sets(text)
    return prog


def _as_bin(text):
    # unit op gop xk xi ximm yk yi yimm zk zi zimm imm dst filt aux imm2 n32: H_INSET -> H_BIN D_INSET with
    # y = the constant imm (the set's address)
    out = []
    for line in text.split("\n"):
        f = line.split()
        if f and f[0] == "unit" and int(f[1]) == H_INSET:
            f[1], f[2], f[6], f[7], f[8] = str(_VM.H_BIN), str(D_INSET), str(_VM.S_IMM), "0", f[12]
            line = " ".join(f)
        out.append(line)
    return "\n".join(out)


class _Lowering:
    """stands in for the native module inside the models: debug_lower records the sets it prints"""

    def __init__(self):
        self.sets = {}

    def debug_lower(self, *args):
        text = _N.debug_lower(*args)
        self.sets.update(parse_sets(text))
        return _as_bin(text)

    def __getattr__(self, name):
        return getattr(_N, name)


@contextlib.contextmanager
def _with_sets():
    low, binop, native = _Lowering(), _VM._binop, _VM.N

    def _binop(op, a, b, valid):
        if op == D_INSET:
            return in_set(low.sets, int(b[0]), a, valid) if len(b) else np.zeros(0, dtype=np.int64)
        return binop(op, a, b, valid)
    _VM._binop, _VM.N = _binop, low
    try:
        yield
    finally:
        _VM._binop, _VM.N = binop, native


def run_pipeline_vm(*args, **kw):
    with _with_sets():
        return _VM.run_pipeline_vm(*args, **kw)


def run_pipeline_device(*args, **kw):
    with _with_sets():
        return _VM.run_pipeline_device(*args, **kw)
