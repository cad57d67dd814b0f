"""ctypes binding of include/resql_b200.h (the drop-in C ABI). No fallback: if the shared
library cannot be loaded, or no sm_100 device is present, every call raises EngineError."""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

RQ_I8, RQ_I32, RQ_I64, RQ_STR = 1, 2, 3, 4
RQ_HOST_PTR, RQ_DEVICE_PTR, RQ_BORROW = 0, 1, 2
SQL_VARCHAR, SQL_CHAR, SQL_BOOL, SQL_INT, SQL_BIGINT, SQL_DECIMAL, SQL_FLOAT, SQL_DATE = range(8)
RQ_PLAN_SHARDED = 1
RQ_PLAN_PARTITIONED = 2


def lib_path():
    return os.path.join(_HERE, "libresql_b200.so")


class EngineError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"resql_b200 error {code}: {msg}")
        self.code = code


class rq_column(C.Structure):
    _fields_ = [("type", C.c_int32), ("width", C.c_int32), ("data", C.c_void_p)]


class rq_node(C.Structure):
    _fields_ = [("op", C.c_int32), ("a", C.c_int32), ("b", C.c_int32), ("c", C.c_int32),
                ("imm", C.c_int64)]


class rq_value(C.Structure):
    _fields_ = [("node", C.c_int32), ("kind", C.c_int32), ("sql_type", C.c_int32),
                ("width", C.c_int32)]


class rq_pipeline(C.Structure):
    _fields_ = [("source_kind", C.c_int32), ("source_id", C.c_int32),
                ("n_nodes", C.c_int32), ("nodes", C.POINTER(rq_node)),
                ("n_args", C.c_int32), ("args", C.POINTER(C.c_int32)),
                ("sink_kind", C.c_int32),
                ("n_keys", C.c_int32), ("keys", C.POINTER(rq_value)),
                ("n_vals", C.c_int32), ("vals", C.POINTER(rq_value)),
                ("size_hint", C.c_int64), ("source_id2", C.c_int32), ("reserved", C.c_int32)]


class rq_order_key(C.Structure):
    _fields_ = [("column", C.c_int32), ("ascending", C.c_int32)]


class rq_plan(C.Structure):
    _fields_ = [("n_tables", C.c_int32), ("tables", C.POINTER(C.c_void_p)),
                ("n_pipelines", C.c_int32), ("pipelines", C.POINTER(rq_pipeline)),
                ("n_order", C.c_int32), ("order", C.POINTER(rq_order_key)),
                ("limit", C.c_int64),
                ("strpool", C.c_char_p), ("strpool_bytes", C.c_int64),
                ("flags", C.c_int32)]


class rq_result_col(C.Structure):
    _fields_ = [("type", C.c_int32), ("width", C.c_int32), ("sql_type", C.c_int32),
                ("sql_width", C.c_int32), ("data", C.c_void_p)]


class rq_result(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("n_cols", C.c_int32), ("cols", C.POINTER(rq_result_col))]


class rq_timings(C.Structure):
    _fields_ = [("lower_ms", C.c_double), ("h2d_ms", C.c_double), ("kernel_ms", C.c_double),
                ("nccl_ms", C.c_double), ("d2h_ms", C.c_double), ("scan_kernel_ms", C.c_double),
                ("kernel_launches", C.c_int32), ("host_syncs", C.c_int32), ("fact_scan_ms", C.c_double)]


class Timings:
    def __init__(self, t):
        for name, _ in rq_timings._fields_:
            setattr(self, name, getattr(t, name))

    def __repr__(self):
        return "Timings(" + ", ".join(f"{k}={getattr(self, k):.4g}" for k, _ in rq_timings._fields_) + ")"


class Result:
    """Columns as numpy arrays in the reference's physical widths, plus SQL types."""

    def __init__(self, columns, sql_types, sql_widths, names=None):
        self.columns = columns
        self.sql_types = sql_types
        self.sql_widths = sql_widths
        self.names = names
        self.n_rows = len(columns[0]) if columns else 0


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise EngineError(-1, f"{p} not built; run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(p)
    lib.rq_last_error.restype = C.c_char_p
    lib.rq_stream.restype = C.c_void_p
    lib.rq_init.argtypes = [C.c_int]
    lib.rq_set_option.argtypes = [C.c_char_p, C.c_double]
    lib.rq_table_upload.argtypes = [C.c_char_p, C.c_int32, C.POINTER(rq_column), C.c_int64,
                                    C.c_int32, C.POINTER(C.c_void_p)]
    lib.rq_table_upload_rows.argtypes = [C.c_char_p, C.c_int32, C.POINTER(C.c_int32),
                                         C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int32,
                                         C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t),
                                         C.POINTER(C.c_void_p)]
    lib.rq_table_alloc.argtypes = [C.c_char_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int64,
                                   C.POINTER(C.c_void_p)]
    lib.rq_table_broadcast.argtypes = [C.c_void_p, C.c_int32]
    lib.rq_table_load_tbl.argtypes = [C.c_char_p, C.c_char_p, C.c_char, C.c_int32, C.POINTER(C.c_int32),
                                      C.POINTER(C.c_int32), C.POINTER(C.c_void_p)]
    lib.rq_table_rows.argtypes = [C.c_void_p]
    lib.rq_table_rows.restype = C.c_int64
    lib.rq_table_free.argtypes = [C.c_void_p]
    lib.rq_plan_execute.argtypes = [C.POINTER(rq_plan), C.POINTER(C.POINTER(rq_result)),
                                    C.POINTER(rq_timings)]
    lib.rq_result_free.argtypes = [C.POINTER(rq_result)]
    lib.rq_dist_unique_id.argtypes = [C.POINTER(C.c_uint8)]
    lib.rq_dist_init.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_uint8)]
    lib.rq_debug_lower.argtypes = [C.POINTER(rq_plan), C.c_int, C.c_int, C.POINTER(C.c_int32),
                                   C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                   C.c_int, C.c_char_p, C.c_int64]
    _lib = lib
    return lib


def debug_lower(plan, pipeline, impl, col_types, col_widths, col_min=None, col_max=None):
    """Host-side lowering of one pipeline to the device program, as text (no GPU needed).
    col_min/col_max: optional per-column value bounds (the upload statistics)."""
    lib = load()

    class _T:
        def __init__(self, names):
            self.names, self.handle = names, None
    tables = {t["name"]: _T(t["columns"]) for t in plan.tables}
    cplan, keep = plan.to_c(tables, 0)
    n = len(col_types)
    ty = (C.c_int32 * n)(*col_types)
    wi = (C.c_int32 * n)(*col_widths)
    mn = (C.c_int64 * n)(*col_min) if col_min is not None else None
    mx = (C.c_int64 * n)(*col_max) if col_max is not None else None
    size = 1 << 16
    while True:       # (long IN lists print one line per set member)
        buf = C.create_string_buffer(size)
        rc = lib.rq_debug_lower(C.byref(cplan), pipeline, impl, ty, wi, mn, mx, n, buf, len(buf))
        if rc == 0:
            return buf.value.decode()
        msg = lib.rq_last_error().decode()
        if "buffer too small" not in msg or size >= 1 << 30:
            raise EngineError(rc, msg)
        size *= 4


ABI_SYMBOLS = ["rq_init", "rq_shutdown", "rq_last_error", "rq_stream", "rq_set_option", "rq_dist_unique_id",
               "rq_dist_init", "rq_table_upload", "rq_table_upload_rows", "rq_table_alloc", "rq_table_broadcast", "rq_table_load_tbl", "rq_table_rows",
               "rq_table_free", "rq_plan_execute", "rq_result_free"]

_NP_OF = {RQ_I8: np.uint8, RQ_I32: np.int32, RQ_I64: np.int64}


def _phys(arr):
    """numpy array -> (rq type, width)."""
    if arr.dtype == np.uint8 and arr.ndim == 1:
        return RQ_I8, 1
    if arr.dtype == np.int32:
        return RQ_I32, 4
    if arr.dtype == np.int64:
        return RQ_I64, 8
    if arr.dtype.kind == "S":
        return RQ_STR, arr.dtype.itemsize
    if arr.dtype == np.uint8 and arr.ndim == 2:
        return RQ_STR, arr.shape[1]
    raise TypeError(f"unsupported column dtype {arr.dtype}")


class Table:
    def __init__(self, handle, names, keepalive=None):
        self.handle = handle
        self.names = list(names)
        self._keep = keepalive

    def rows(self):
        return load().rq_table_rows(self.handle)

    def free(self):
        if self.handle:
            load().rq_table_free(self.handle)
            self.handle = None


class Engine:
    """One engine per process / GPU (mirrors the single-caller reference, execute.h:509)."""

    def __init__(self, device=0):
        self.lib = load()
        self._check(self.lib.rq_init(int(device)))
        self.device = device

    def _check(self, rc):
        if rc != 0:
            raise EngineError(rc, self.lib.rq_last_error().decode("utf-8", "replace"))

    def shutdown(self):
        self.lib.rq_shutdown()

    def stream(self):
        return self.lib.rq_stream()

    def set_option(self, key, value):
        self._check(self.lib.rq_set_option(key.encode(), float(value)))

    # -- multi-GPU --------------------------------------------------------------------------
    def dist_unique_id(self):
        buf = (C.c_uint8 * 128)()
        self._check(self.lib.rq_dist_unique_id(buf))
        return bytes(buf)

    def dist_init(self, rank, world, uid):
        buf = (C.c_uint8 * 128).from_buffer_copy(uid)
        self._check(self.lib.rq_dist_init(rank, world, buf))

    # -- tables -----------------------------------------------------------------------------
    def upload(self, name, columns):
        """columns: ordered dict name -> numpy array (host) in the reference's physical type:
        uint8 (BOOL/CHAR(1)), int32 (INT/DATE), int64 (BIGINT/DECIMAL), 'S<n+1>' (CHAR/VARCHAR)."""
        names = list(columns.keys())
        cols = (rq_column * len(names))()
        keep = []
        n_rows = None
        for i, nm in enumerate(names):
            a = np.ascontiguousarray(columns[nm])
            t, w = _phys(a)
            keep.append(a)
            cols[i].type, cols[i].width = t, w
            cols[i].data = a.ctypes.data
            n = a.shape[0]
            if n_rows is None:
                n_rows = n
            elif n != n_rows:
                raise ValueError("ragged columns")
        h = C.c_void_p()
        self._check(self.lib.rq_table_upload(name.encode(), len(names), cols, n_rows, RQ_HOST_PTR, C.byref(h)))
        return Table(h, names)

    def upload_device(self, name, columns, n_rows, borrow=True):
        """columns: ordered dict name -> (device_ptr:int, rq_type, width). With borrow=True the
        caller keeps the buffers alive (e.g. torch tensors) and they are used in place."""
        names = list(columns.keys())
        cols = (rq_column * len(names))()
        for i, nm in enumerate(names):
            ptr, t, w = columns[nm]
            cols[i].type, cols[i].width, cols[i].data = t, w, ptr
        h = C.c_void_p()
        flags = RQ_DEVICE_PTR | (RQ_BORROW if borrow else 0)
        self._check(self.lib.rq_table_upload(name.encode(), len(names), cols, n_rows, flags, C.byref(h)))
        return Table(h, names, keepalive=columns)

    def alloc(self, name, schema, n_rows):
        """empty table: schema = ordered dict name -> (rq_type, width); filled by broadcast()"""
        names = list(schema.keys())
        ty = (C.c_int32 * len(names))(*[schema[n][0] for n in names])
        wi = (C.c_int32 * len(names))(*[schema[n][1] for n in names])
        h = C.c_void_p()
        self._check(self.lib.rq_table_alloc(name.encode(), len(names), ty, wi, n_rows, C.byref(h)))
        return Table(h, names)

    def broadcast(self, table, root=0):
        """collective: every rank's `table` gets the contents of rank `root`'s (NVLink, ncclBroadcast)"""
        self._check(self.lib.rq_table_broadcast(table.handle, root))
        return table

    def upload_replicated(self, name, columns, root=0, rank=0):
        """columns (host numpy, as for upload) are read on `root` only; other ranks only use dtype / shape"""
        if rank == root:
            t = self.upload(name, columns)
        else:
            schema = {n: _phys(np.asarray(a)) for n, a in columns.items()}
            t = self.alloc(name, schema, len(next(iter(columns.values()))))
        return self.broadcast(t, root)

    def load_tbl(self, name, path, schema, terminator="|"):
        """parallel text loader; schema = ordered [(column, RQ_SQL_* type, n of CHAR(n)/VARCHAR(n) or 0)]"""
        n = len(schema)
        ty = (C.c_int32 * n)(*[s[1] for s in schema])
        wi = (C.c_int32 * n)(*[s[2] for s in schema])
        h = C.c_void_p()
        self._check(self.lib.rq_table_load_tbl(name.encode(), str(path).encode(), terminator.encode(), n, ty, wi, C.byref(h)))
        return Table(h, [s[0] for s in schema])

    def upload_rows(self, name, names, types, widths, offsets, tuple_size, blocks):
        """Row-store upload (reference DataBlocks): blocks = list of bytes-like objects."""
        n = len(names)
        ty = (C.c_int32 * n)(*types)
        wi = (C.c_int32 * n)(*widths)
        of = (C.c_int32 * n)(*offsets)
        keep = [np.frombuffer(b, dtype=np.uint8) for b in blocks]
        ptrs = (C.c_void_p * len(keep))(*[k.ctypes.data for k in keep])
        sizes = (C.c_size_t * len(keep))(*[k.size for k in keep])
        h = C.c_void_p()
        self._check(self.lib.rq_table_upload_rows(name.encode(), n, ty, wi, of, tuple_size,
                                                  len(keep), ptrs, sizes, C.byref(h)))
        return Table(h, names)

    # -- execution --------------------------------------------------------------------------
    def execute(self, plan, tables, flags=0):
        """plan: resql_b200.plan.Plan; tables: dict name -> Table. Returns (Result, Timings)."""
        # the flat C plan is built once per (plan, table handles, flags): a repeated query costs no
        # Python-side marshalling (the reference likewise re-runs a prepared plan)
        key = (flags,) + tuple((t["name"], tables[t["name"]].handle.value) for t in plan.tables)
        cache = plan.__dict__.setdefault("_c_cache", {})
        if key not in cache:
            if len(cache) > 16:
                cache.clear()
            cache[key] = plan.to_c(tables, flags)
        cplan, keep = cache[key]
        res = C.POINTER(rq_result)()
        tm = rq_timings()
        self._check(self.lib.rq_plan_execute(C.byref(cplan), C.byref(res), C.byref(tm)))
        try:
            r = res.contents
            cols, st, sw = [], [], []
            for c in range(r.n_cols):
                rc = r.cols[c]
                n = r.n_rows
                if rc.type == RQ_STR:
                    raw = np.ctypeslib.as_array(C.cast(rc.data, C.POINTER(C.c_uint8)), shape=(max(n, 1) * rc.width,))
                    arr = raw[: n * rc.width].copy().view(f"S{rc.width}")
                else:
                    dt = _NP_OF[rc.type]
                    raw = np.ctypeslib.as_array(C.cast(rc.data, C.POINTER(C.c_uint8)), shape=(max(n, 1) * rc.width,))
                    arr = raw[: n * rc.width].copy().view(dt)
                cols.append(arr)
                st.append(rc.sql_type)
                sw.append(rc.sql_width)
        finally:
            self.lib.rq_result_free(res)
        return Result(cols, st, sw, plan.result_names), Timings(tm)
