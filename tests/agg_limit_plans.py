"""Grouped-aggregation plans and an exact restatement of the host rules that the scan kernel's exactness
rests on, for test_lowering_aggmodes.py and test_gpu_agg_limits.py: value bounds (Lowerer::derive_bounds
in engine.cu), the register path's SUM accumulation modes and flush bound (choose_agg_modes) and the
packed group key (pack_group_key, engine_exec.inl). Python integers throughout. Test infrastructure only."""
from inlist_plans import Pipe, new_plan, SINK_AGG
from plan_fuzz import SQL_CHAR, SQL_INT, SQL_BIGINT, AGG_SUM, AGG_COUNT, AGG_MIN, AGG_MAX

KR = 8                        # tuples per lane per tile (rq_internal.h kR)
TILE = 32 * KR
I64_MIN, I64_MAX = -2 ** 63, 2 ** 63 - 1
I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1
AM_FULL, AM_P1, AM_P2, AM_W64 = 0, 1, 2, 3
RQ_I8, RQ_I32, RQ_I64 = 1, 2, 3
IMPL_LOWAGG, IMPL_REGAGG = 1, 5
SWAP = {"LT": "GT", "LE": "GE", "GT": "LT", "GE": "LE", "EQ": "EQ"}


# ---- interval rules (derive_bounds) ------------------------------------------------------------------
def col_bounds(rq_type, stats):
    """bounds of a source column: its upload statistics (lo, hi), else what its physical type allows"""
    if stats is not None and stats[0] <= stats[1]:
        return stats
    return {RQ_I8: (0, 255), RQ_I32: (I32_MIN, I32_MAX)}.get(rq_type, (I64_MIN, I64_MAX))


def narrow(lo, hi, filters):
    """the bounds of a column seen by the sink, given the `col CMP const` filters on it: (op, const,
    const_on_left). No tuple passes contradictory filters; any bounds do then, the rule takes the
    narrowed low bound (or the high one when no filter raised the low bound)."""
    clo, chi = I64_MIN, I64_MAX
    for op, k, left in filters:
        op = SWAP[op] if left else op
        if op == "LT":
            chi = min(chi, k - 1)
        elif op == "LE":
            chi = min(chi, k)
        elif op == "GT":
            clo = max(clo, k + 1)
        elif op == "GE":
            clo = max(clo, k)
        else:
            clo, chi = max(clo, k), min(chi, k)
    lo, hi = max(lo, clo), min(hi, chi)
    if lo > hi:
        lo = hi = clo if clo > I64_MIN else chi
    return max(lo, I64_MIN), min(hi, I64_MAX)


def clamp(lo, hi):
    """a result that may wrap around int64 is unknown"""
    return (lo, hi) if I64_MIN <= lo and hi <= I64_MAX else (I64_MIN, I64_MAX)


def add(a, b):
    return clamp(a[0] + b[0], a[1] + b[1])


def sub(a, b):
    return clamp(a[0] - b[1], a[1] - b[0])


def mul(a, b):
    c = [x * y for x in a for y in b]
    return clamp(min(c), max(c))


def select(b, c):
    return min(b[0], c[0]), max(b[1], c[1])


# ---- SUM accumulation modes and the flush bound (choose_agg_modes) ----------------------------------
def bound_tiles(piece_max):
    """tiles a lane may add kR values of at most piece_max each before a 32-bit sum could wrap"""
    return (2 ** 32 - 1) // (KR * max(piece_max, 1))


def agg_mode(kind, lo, hi):
    """(mode, P2 shift, the largest value of each 32-bit piece sum) of one aggregate over [lo, hi]"""
    if kind != AGG_SUM or lo < 0:
        return AM_FULL, 0, []
    if hi < 2 ** 25:
        return AM_P1, 0, [hi]
    if hi < 2 ** 32:
        return AM_W64, 0, []
    if hi < 2 ** 48:
        sh = (hi.bit_length() + 1) // 2
        return AM_P2, sh, [2 ** sh - 1, hi >> sh]
    return AM_FULL, 0, []


def flush_bound(aggs):
    """aggs: [(kind, lo, hi)] -> the flush bound in tiles; the 32-bit tuple counters count 1 a tuple"""
    pieces = [p for kind, lo, hi in aggs for p in agg_mode(kind, lo, hi)[2]]
    return min(bound_tiles(p) for p in pieces + [1])


def tiles_per_warp(rows, warps, sms=148):
    tiles = max(1, -(-rows // TILE))
    grid = min(-(-tiles // warps), sms)
    return -(-tiles // (grid * warps))


# ---- packed group key (pack_group_key) ---------------------------------------------------------------
def key_field(lo, hi, width=None):
    """(bits, sign) of one key: a column key starts from its physical width (unsigned for 1 byte), any
    other value from 64 signed bits; a key proven non-negative takes only the bits its bound needs"""
    bits, sign = (8 * width, int(width != 1)) if width else (64, 1)
    if lo >= 0:
        need = max(1, min(63, hi.bit_length()))
        if need < bits:
            bits, sign = need, 0
    return bits, sign


def pack_keys(fields):
    """[(bits, sign)] -> ([(shift, bits, sign)], key32), or None when the key needs more than 64 bits"""
    out, total = [], 0
    for bits, sign in fields:
        if total + bits > 64:
            return None
        out.append((total, bits, sign))
        total += bits
    return out, int(total <= 31)


# ---- what rq_debug_lower prints ------------------------------------------------------------------------
def parse_lowering(text):
    r = {"aggmode": {}, "keyfield": {}, "agg": {}, "aggmap": {}}
    for line in text.splitlines():
        f = line.split()
        if f[0] == "cols":
            r["warps"], r["stages"] = int(f[f.index("warps") + 1]), int(f[f.index("stages") + 1])
            r["packed"] = int(f[f.index("packed") + 1])
        elif f[0] in ("aggmode", "keyfield", "agg", "aggmap"):
            r[f[0]][int(f[1])] = tuple(int(x) for x in f[2:])
        elif f[0] in ("flushbound", "key32", "lowagg_groups"):
            r[f[0]] = int(f[1])
    return r


def lower(d, impl, types, widths, stats=None):
    from resql_b200 import native as N
    from resql_b200.plan import Plan
    mn = [s[0] for s in stats] if stats else None
    mx = [s[1] for s in stats] if stats else None
    return parse_lowering(N.debug_lower(Plan(d), 0, impl, types, widths, mn, mx))


# ---- plans ---------------------------------------------------------------------------------------------
def agg_plan(columns, build):
    """one aggregation pipeline over table t(columns); build(p) -> (keys, vals) with keys [(node, sql
    type)] or [(node, sql type, width)] and vals [(node, kind)] (node None for COUNT(*))"""
    d, pool = new_plan({"t": columns})
    p = Pipe(d, "t", columns, pool)
    keys, vals = build(p)
    p.done(SINK_AGG, [[n if n is not None else 0, kind, SQL_BIGINT, 0] for n, kind in vals],
           [[k[0], 0, k[1], k[2] if len(k) > 2 else 0] for k in keys])
    return d


def cmp_filter(p, node, op, k, left=False):
    c = p.const(k)
    p.filter(p.n(op, c, node) if left else p.n(op, node, c))


def sum_by(columns, keys, value, filters=(), kinds=(AGG_SUM,), key_sql=None):
    """select keys, <kinds>(value), count(*) from t where filters group by keys; value: a column name or
    a function of the Pipe giving a node; filters: [(column, op, const, const_on_left)]; key_sql: key
    column -> (sql type, width), BIGINT by default"""
    def build(p):
        for c, op, k, left in filters:
            cmp_filter(p, p.col(c), op, k, left)
        v = value(p) if callable(value) else p.col(value)
        return ([(p.col(k),) + (key_sql or {}).get(k, (SQL_BIGINT, 0)) for k in keys],
                [(v, kind) for kind in kinds] + [(None, AGG_COUNT)])
    return agg_plan(columns, build)


def wrap64(x):
    """x as a two's-complement int64"""
    x &= 2 ** 64 - 1
    return x - 2 ** 64 if x >= 2 ** 63 else x
