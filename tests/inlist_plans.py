"""Plans with IN lists for the set-unit tests (test_lowering_inlist.py, test_gpu_inlist.py): the OR trees
of equality tests the reference's parser emits for `x IN (c1, ..., ck)`, in every associativity, and
random plans of tests/plan_fuzz.py with such lists injected. Test infrastructure only."""
import random

from plan_fuzz import OP, SQL_CHAR, SQL_VARCHAR, SQL_INT, SQL_BIGINT, random_plan

SINK_AGG, SINK_BUILD, SINK_MAT = 1, 2, 3


class Pipe:
    """One pipeline under construction: postfix nodes over the columns of one table."""

    def __init__(self, plan, table, columns, pool):
        self.plan, self.table, self.columns, self.pool = plan, table, columns, pool
        self.nodes, self.args = [], []

    def n(self, op, a=0, b=0, c=0, imm=0):
        self.nodes.append([OP[op], a, b, c, imm])
        return len(self.nodes) - 1

    def col(self, name):
        return self.n("COL", self.columns.index(name))

    def const(self, v):
        return self.n("CONST", imm=int(v))

    def cstr(self, s):
        off = len(self.pool[0])
        self.pool[0] += (s.decode("latin1") if isinstance(s, bytes) else s) + "\0"
        return self.n("CONST_STR", imm=off)

    def inlist(self, v, consts, shape="right", eq="EQ", const_left=False):
        """OR tree of `v eq c` over consts. right: all leaves first, then OR(e1, OR(e2, ...)) (the
        reference's parser); left: OR(OR(e1, e2), e3) ...; balanced: pairwise."""
        def leaf(c):
            k = self.const(c) if eq == "EQ" else self.cstr(c)
            return self.n(eq, k, v) if const_left else self.n(eq, v, k)
        if shape == "right":
            es = [leaf(c) for c in consts]
            acc = es[-1]
            for e in reversed(es[:-1]):
                acc = self.n("OR", e, acc)
            return acc
        if shape == "left":
            acc = leaf(consts[0])
            for c in consts[1:]:
                acc = self.n("OR", acc, leaf(c))
            return acc
        level = [leaf(c) for c in consts]
        while len(level) > 1:
            nxt = [self.n("OR", level[i], level[i + 1]) for i in range(0, len(level) - 1, 2)]
            if len(level) % 2:
                nxt.append(level[-1])
            level = nxt
        return level[0]

    def filter(self, x):
        return self.n("FILTER", x)

    def done(self, sink, vals, keys=(), source_kind=1, source_id=None):
        sid = [t["name"] for t in self.plan["tables"]].index(self.table) if source_id is None else source_id
        self.plan["pipelines"].append({"source_kind": source_kind, "source_id": sid, "sink_kind": sink, "nodes": self.nodes,
                                       "args": self.args, "keys": [list(k) for k in keys], "vals": [list(v) for v in vals],
                                       "size_hint": 0})
        self.plan["strpool"] = self.pool[0]


def new_plan(tables):
    """tables: {name: [columns]} -> (plan dict, pool cell)"""
    return {"tables": [{"name": t, "columns": list(c)} for t, c in tables.items()], "pipelines": [], "order": [],
            "limit": -1, "strpool": ""}, [""]


def select_in(table, columns, tested, consts, out, shape="right", eq="EQ", const_left=False, computed=False):
    """select <out> from table where <tested> in (consts); out: [(column, sql type, width)].
    computed: the tested value is tested + 1 (a slot operand)."""
    d, pool = new_plan({table: columns})
    p = Pipe(d, table, columns, pool)
    v = p.col(tested)
    if computed:
        v = p.n("ADD", v, p.const(1))
    p.filter(p.inlist(v, consts, shape, eq, const_left))
    p.done(SINK_MAT, [[p.col(c), 0, t, w] for c, t, w in out])
    return d


def case_in(table, columns, tested, consts, other, shape="right", eq="EQ"):
    """select case when tested in (consts) then other else 0 end, tested from table"""
    d, pool = new_plan({table: columns})
    p = Pipe(d, table, columns, pool)
    v = p.col(tested)
    sel = p.n("SELECT", p.inlist(v, consts, shape, eq), p.col(other), p.const(0))
    p.done(SINK_MAT, [[sel, 0, SQL_BIGINT, 0], [p.col(other), 0, SQL_BIGINT, 0]])
    return d


def two_lists(table, columns, a, ka, b, kb, out):
    """select out from table where a in (ka) or b in (kb)"""
    d, pool = new_plan({table: columns})
    p = Pipe(d, table, columns, pool)
    p.filter(p.n("OR", p.inlist(p.col(a), ka), p.inlist(p.col(b), kb, "left")))
    p.done(SINK_MAT, [[p.col(c), 0, t, w] for c, t, w in out])
    return d


def sum_in(table, columns, tested, consts, summed, eq="EQ", group=None):
    """select [group,] sum(summed), count(*) from table where tested in (consts) [group by group]"""
    d, pool = new_plan({table: columns})
    p = Pipe(d, table, columns, pool)
    p.filter(p.inlist(p.col(tested), consts, "right", eq))
    keys = [[p.col(group), 0, SQL_INT, 0]] if group else []
    p.done(SINK_AGG, [[p.col(summed), 1, SQL_BIGINT, 0], [0, 2, SQL_BIGINT, 0]], keys)
    return d


# ---- random plans with IN lists ---------------------------------------------------------------------
def _int_consts(rng, k):
    pool = [rng.randint(1, 7), rng.randint(1, 200), rng.randint(-5, 70000), rng.randint(1, 60000), 2 ** 40, -3]
    return [rng.choice(pool) if rng.random() < 0.2 else rng.randint(-2, 60000) for _ in range(k)]


def random_inlist_plan(seed):
    """plan_fuzz.random_plan(seed) with an IN filter or an IN-in-CASE value added to its first pipeline
    that scans a table with an integer or string column"""
    rng = random.Random(seed * 7919 + 1)
    d = random_plan(seed)
    pool = [d.get("strpool", "")]
    for pl in d["pipelines"]:
        if pl["source_kind"] != 1:
            continue
        cols = d["tables"][pl["source_id"]]["columns"]
        p = Pipe(d, d["tables"][pl["source_id"]]["name"], cols, pool)
        p.nodes, p.args = pl["nodes"], pl["args"]
        ints = [c for c in cols if c in ("l_orderkey", "l_partkey", "l_linenumber", "o_custkey", "o_orderkey", "c_custkey",
                                         "c_nationkey", "o_shippriority", "l_quantity", "l_returnflag", "o_orderstatus")]
        strs = [c for c in cols if c in ("l_shipmode", "l_shipinstruct", "o_orderpriority", "c_mktsegment")]
        k = rng.choice([1, 2, 3, 5, 11, 12, 40, 300])
        shape = rng.choice(["right", "left", "balanced"])
        if strs and (not ints or rng.random() < 0.4):
            c = rng.choice(strs)
            words = ["MAIL", "SHIP", "AIR", "RAIL", "TRUCK", "FOB", "REG AIR", "NONE", "COLLECT COD", "DELIVER IN PERSON",
                     "TAKE BACK RETURN", "1-URGENT", "2-HIGH", "5-LOW", "BUILDING", "MACHINERY", "", "AIR  ", "MAIL "]
            consts = [rng.choice(words) for _ in range(k)]
            eq = rng.choice(["EQ_CHAR", "EQ_VARCHAR"])
            v = p.col(c)
        elif ints:
            c = rng.choice(ints)
            consts = _int_consts(rng, k) if c not in ("l_returnflag", "o_orderstatus") else [rng.choice(b"ANRFOP") for _ in range(k)]
            eq = "EQ"
            v = p.col(c)
        else:
            continue
        tree = p.inlist(v, consts, shape, eq, const_left=(eq == "EQ" and rng.random() < 0.3))
        if rng.random() < 0.6:
            p.filter(tree)
        elif pl["sink_kind"] == SINK_MAT:
            sel = p.n("SELECT", tree, p.const(rng.randint(1, 9)), p.const(0))
            pl["vals"].append([sel, 0, SQL_BIGINT, 0])
            _widen_result(d, pl)
        else:
            p.filter(tree)
        break
    d["strpool"] = pool[0]
    return d


def _widen_result(d, pl):
    if pl is d["pipelines"][-1]:
        for key in ("result_names", "result_types"):
            if key in d:
                d[key] = d[key] + ([f"in{len(pl['vals'])}"] if key == "result_names" else [[SQL_BIGINT, 0]])


__all__ = ["Pipe", "new_plan", "select_in", "case_in", "two_lists", "sum_in", "random_inlist_plan", "SQL_CHAR",
           "SQL_VARCHAR", "SQL_INT", "SQL_BIGINT", "SINK_AGG", "SINK_BUILD", "SINK_MAT"]
