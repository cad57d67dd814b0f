/*
 * resql_b200 - C ABI of the B200-native execution engine for ReSQL query pipelines.
 *
 * This is the drop-in boundary. The reference (Henning1/resql) has no FFI; its seam is the C++
 * span inside executeSelectPlan (src/execute.h:213-247):
 *
 *     JitContextFlounder ctx(config.jit);  root->produceFlounder(ctx, {});      execute.h:229-232
 *     ctx.compile();  ctx.execute();                                            execute.h:233,240
 *     root->retrieveResult();                                                   execute.h:241
 *
 * A host shim compiled inside the reference's single translation unit (resql_b200/host/
 * gpu_executor.h, see INTEGRATION.md) walks the typed operator tree, lowers it to the flat plan
 * below and calls these entry points instead of the Flounder/asmjit JIT. The library is built by
 * nvcc alone, never sees a reference header, throws nothing across the ABI, and owns all device
 * memory. Every call returns an int status (0 = RQ_OK); rq_last_error() gives the message the
 * shim rethrows as ResqlError (src/util/ResqlError.h; reference error path execute.h:536-541).
 *
 * Threading: one caller thread per process, one process per GPU (the reference is likewise
 * single-caller: execute.h:509 is invoked from the REPL / select() loop only).
 *
 * Value model (mirrors src/types.h:213-261 and src/values.h:15-24): every scalar the plan
 * computes is a 64-bit integer. INT/DATE (4 B in the reference tuple) are sign-extended on
 * load, BOOL/CHAR(1) (1 B) zero-extended, BIGINT/DECIMAL are int64 (DECIMAL(p,s) = value*10^s,
 * wrap-around arithmetic, ExpressionsJitFlounder.h:298-402). CHAR(n>1)/VARCHAR(n) values are
 * device addresses of NUL-terminated bytes, i.e. "strings by reference" exactly like the
 * reference's hash-table layout (ValuesJitFlounder.h:192); they are copied by value only into
 * the final result (ValuesJitFlounder.h:195, materialize.h:78-220).
 */
#ifndef RESQL_B200_H
#define RESQL_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ---------------------------------------------------------------------- */
#define RQ_OK               0
#define RQ_ERR_INVALID      1   /* malformed plan / argument                                  */
#define RQ_ERR_CUDA         2   /* CUDA runtime failure (message has the CUDA error string)   */
#define RQ_ERR_UNSUPPORTED  3   /* plan shape outside the implemented hot path                */
#define RQ_ERR_NOT_INIT     4
#define RQ_ERR_NCCL         5
#define RQ_ERR_RUNTIME      6   /* data-dependent failure (e.g. division by zero: the
                                   reference dies with SIGFPE, ExpressionsJitFlounder.h:408) */

/* ---- physical column types (reference widths: src/types.h:213-261) ---------------------- */
#define RQ_I8   1   /* BOOL, CHAR(1): payload byte (the reference stores CHAR(1) as byte+NUL)  */
#define RQ_I32  2   /* INT, DATE (yyyymmdd)                                                    */
#define RQ_I64  3   /* BIGINT, DECIMAL(p,s)                                                    */
#define RQ_STR  4   /* CHAR(n>1), VARCHAR(n): width = n+1 bytes per row, NUL-terminated,
                       not space padded (values.h:151-198)                                     */

/* logical SQL type tags carried through to the result (src/types.h:66-76 order) */
#define RQ_SQL_VARCHAR 0
#define RQ_SQL_CHAR    1
#define RQ_SQL_BOOL    2
#define RQ_SQL_INT     3
#define RQ_SQL_BIGINT  4
#define RQ_SQL_DECIMAL 5
#define RQ_SQL_FLOAT   6
#define RQ_SQL_DATE    7

/* ---- lifecycle -------------------------------------------------------------------------- */
/* Replaces construction of JitContextFlounder (JitContextFlounder.h:182-236). `device` is the
 * CUDA ordinal of this process's GPU. */
int rq_init(int device);
int rq_shutdown(void);
const char* rq_last_error(void);
/* cudaStream_t the engine launches on (so a harness can bracket it with its own events). */
void* rq_stream(void);
/* Engine knobs, the counterpart of the reference's control variables (`threads=4`, `emitmc=true`;
 * processControl, execute.h:454-474). Keys: "split_min_rows", "split_frac" (two-pass probes),
 * "prune_builds", "topk", "replay", "graphs", "direct_joins" (0/1), "stages", "warps" (scan-kernel layout, 0 = automatic),
 * "trace" (0/1), "late_materialize" (0 never, 1 = default: materialize pipelines wider than the early form
 * holds - more than 24 outputs, 16 staged columns, 12 live values or 8 string columns - write row / entry
 * references and gather their columns afterwards, up to 64 columns; 2: that form wherever it applies),
 * "in_lists" (OR trees of equality tests of one value against constants as one set test: 0 never, keeping
 * one compare per value; 1 = default: integer lists of 2 values or more, string lists of 4 or more;
 * 2: every list of 2 values or more),
 * "sink_rounds" (materialize pipelines whose computed outputs need more than 12 live values store them in
 * rounds that each fit, up to 64 outputs: 0 never; 1 = default: only where the single sink cannot hold
 * the values; 2: wherever it applies).
 * Defaults are the production choices; the parity tests force rarely taken paths. */
int rq_set_option(const char* key, double value);

/* Multi-GPU (one process per GPU). rank 0 calls rq_dist_unique_id, the harness broadcasts the
 * 128 bytes (torch.distributed / MPI / file), every rank calls rq_dist_init. After that, plans
 * executed with RQ_PLAN_SHARDED exchange the per-rank result of the last aggregation (NCCL
 * all-gather of the group tables) and re-aggregate it on every rank (SUM/COUNT partials add,
 * MIN/MAX take min/max) before AVG finalisation, ORDER BY and LIMIT; a plan without aggregation
 * concatenates the per-rank relations. The table scanned by that aggregation's pipeline holds
 * this rank's row range, all other tables are complete on every rank. */
int rq_dist_unique_id(uint8_t out_id[128]);
int rq_dist_init(int rank, int world_size, const uint8_t id[128]);

/* ---- tables (replaces the execution-time use of the row store, dbdata.h:105-461) --------- */
typedef struct rq_table rq_table;

typedef struct {
    int32_t     type;      /* RQ_I8 / RQ_I32 / RQ_I64 / RQ_STR                                 */
    int32_t     width;     /* bytes per row: 1, 4, 8, or n+1 for RQ_STR                        */
    const void* data;      /* n_rows * width bytes (host pointer, or device if RQ_DEVICE_PTR)  */
} rq_column;

#define RQ_HOST_PTR     0
#define RQ_DEVICE_PTR   1   /* columns already live on this GPU; copied device-to-device       */
#define RQ_BORROW       2   /* with RQ_DEVICE_PTR: do not copy, caller keeps buffers alive     */

/* Columnar upload. Host buffers are borrowed for the duration of the call only. */
int rq_table_upload(const char* name, int32_t n_cols, const rq_column* cols, int64_t n_rows,
                    int32_t flags, rq_table** out);

/* Row-store upload: transposes the reference's DataBlocks (dbdata.h:23-102; packed NSM tuples,
 * tuple_size = Schema::_tupSize, offsets = Schema::getOffsetInTuple, schema.h:94-106) into
 * device columns on the GPU. This is the hook for executeBulkInsert (execute.h:332-388).
 * For CHAR(1) pass type RQ_I8 and the offset of the payload byte. */
int rq_table_upload_rows(const char* name, int32_t n_cols, const int32_t* types,
                         const int32_t* widths, const int32_t* offsets, int32_t tuple_size,
                         int32_t n_blocks, const uint8_t* const* blocks,
                         const size_t* block_bytes, rq_table** out);
/* Parallel text loader: parses a `.tbl` file (one row per line, every field followed by `terminator`)
 * straight into a device-resident table; replaces the row-store fill of executeBulkInsert
 * (execute.h:332-388; field semantics of parse*Constant, expressions.h:369-455, incl. DECIMAL = the
 * literal's digits with the point removed and DATE yyyy-mm-dd / yyyy/mm/dd). The text crosses PCIe in
 * segments cut at line ends; the GPU finds the line starts and parses one row per thread.
 * sql_types[] = RQ_SQL_*, sql_widths[] = n of CHAR(n) / VARCHAR(n) (ignored for other types). */
int rq_table_load_tbl(const char* name, const char* path, char terminator, int32_t n_cols,
                      const int32_t* sql_types, const int32_t* sql_widths, rq_table** out);

/* Replicated tables on several GPUs (the build sides of a sharded plan: "small build sides are
 * NCCL-broadcast over NVLink", north_star). One rank uploads the table from its host (rq_table_upload /
 * rq_table_upload_rows); every other rank creates an empty table of the same schema and row count with
 * rq_table_alloc; then ALL ranks call rq_table_broadcast (collective, after rq_dist_init): the
 * contents of `root`'s table replace the others' over NVLink (ncclBroadcast of the column storage),
 * and every rank takes the column statistics of its copy. N ranks cost one host upload instead of N.
 * The reference has no counterpart (one process, one row store: dbdata.h:105-461). */
int rq_table_alloc(const char* name, int32_t n_cols, const int32_t* types, const int32_t* widths,
                   int64_t n_rows, rq_table** out);
int rq_table_broadcast(rq_table* t, int32_t root);

int64_t rq_table_rows(const rq_table* t);
int rq_table_free(rq_table* t);

/* ---- plan: typed postfix programs ------------------------------------------------------- */
/* One node = one entry of a postfix (dependency-ordered) program; operands refer to EARLIER
 * nodes of the same pipeline by index. Replaces emitExpression
 * (ExpressionsJitFlounder.h:1080-1114) - there is no runtime code generation. */
enum rq_op {
    RQ_OP_COL = 1,      /* a = source column index                      (emitAttribute :886)   */
    RQ_OP_CONST,        /* imm = value                                  (emitConstant :248)    */
    RQ_OP_CONST_STR,    /* imm = byte offset into rq_plan.strpool (NUL-terminated)             */
    RQ_OP_ADD,          /* a + b   wrap-around int64                    (:298-331)             */
    RQ_OP_SUB,          /* a - b                                        (:336-366)             */
    RQ_OP_MUL,          /* a * b   low 64 bits (imul)                   (:371-402)             */
    RQ_OP_DIV,          /* a / b   truncating (cqo; idiv)               (:408-420)             */
    RQ_OP_AND,          /* bitwise on 0/1                               (:446-455)             */
    RQ_OP_OR,           /*                                              (:460-468)
                           An OR tree whose leaves all test one value for equality against constants
                           (EQ, or only EQ_CHAR, or only EQ_VARCHAR; what `x IN (...)` parses to) is
                           evaluated as one set-membership test, with no limit on its length.      */
    RQ_OP_LT, RQ_OP_LE, RQ_OP_GT, RQ_OP_GE,   /* signed compare -> 0/1  (:474-615)             */
    RQ_OP_EQ,           /* integer equality -> 0/1                      (:620-632)             */
    RQ_OP_NEQ,          /* 1 - EQ                                       (:1036-1043)           */
    RQ_OP_EQ_CHAR,      /* compareChar: equal ignoring trailing blanks  (qlib/scalar.h:27-46)  */
    RQ_OP_EQ_VARCHAR,   /* compareVarchar: exact                        (qlib/scalar.h:16-24)  */
    RQ_OP_NEQ_CHAR, RQ_OP_NEQ_VARCHAR,
    RQ_OP_LIKE,         /* stringLikeCheck(a, pattern b)                (qlib/scalar.h:57-120) */
    RQ_OP_SELECT,       /* a ? b : c   (one WHEN/THEN arm of emitCase :720-754)                */
    RQ_OP_FILTER,       /* drop the tuple unless (a & 0xff) != 0        (selection.h:62-66)    */
    RQ_OP_PROBE,        /* a = index of the build pipeline; b = first entry, c = count in
                           rq_pipeline.args (probe key nodes). Drops tuples without a match.
                           imm bit0 = single match (hashjoin.h:168-214) else multi (:118-165);
                           the other imm bits must be 0 (used inside the library)              */
    RQ_OP_PAYLOAD       /* a = PROBE node, b = payload column of that build                    */
};

typedef struct {
    int32_t op;         /* enum rq_op                                                          */
    int32_t a, b, c;    /* operand node indices / column / payload indices (see rq_op)         */
    int64_t imm;
} rq_node;

/* aggregate kinds (aggregation.h:95-152); AVG is split into SUM+COUNT by the caller exactly
 * like AggregationOp::splitAverages (aggregation.h:167-179) and re-merged by a later pipeline
 * with MUL 100 / DIV (getAvgFromSumAndCount :182-204). */
#define RQ_AGG_SUM   1
#define RQ_AGG_COUNT 2
#define RQ_AGG_MIN   3
#define RQ_AGG_MAX   4

#define RQ_SRC_TABLE     1   /* source_id indexes rq_plan.tables                               */
#define RQ_SRC_PIPELINE  2   /* source_id = earlier pipeline whose sink is AGG or MATERIALIZE  */
#define RQ_SRC_CROSS     3   /* cross product of two earlier materialized pipelines, source_id x
                                source_id2 (NestedLoopsJoinOp, nestedloopsjoin.h:5-94: both children
                                are materialized, every pair is produced, an optional condition
                                follows as RQ_OP_FILTER). The pairs are streamed through the scan
                                kernel, never materialized; just under 2^40 pairs at most
                                (RQ_ERR_UNSUPPORTED beyond). COL indices address the columns of source_id first, then
                                those of source_id2.                                             */

#define RQ_SRC_ONE_ROW   4   /* a single tuple without attributes: leaf projection, "creates a
                                single-line table from constants" (projection.h:49-58, `select 1+1`) */

#define RQ_SINK_AGG          1   /* GROUP BY keys + aggregates (aggregation.h:240-295)          */
#define RQ_SINK_BUILD        2   /* hash-join build: keys + payload (hashjoin.h:226-256)        */
#define RQ_SINK_MATERIALIZE  3   /* append tuples to an output relation (materialize.h:78)     */

typedef struct {
    int32_t node;        /* node that yields the value                                         */
    int32_t kind;        /* AGG sinks, aggregate entries: RQ_AGG_*; otherwise 0                */
    int32_t sql_type;    /* RQ_SQL_* (for the result schema / string semantics)                */
    int32_t width;       /* CHAR/VARCHAR: n; DECIMAL: precision<<8 | scale; else 0             */
} rq_value;

typedef struct {
    int32_t         source_kind;
    int32_t         source_id;
    int32_t         n_nodes;
    const rq_node*  nodes;
    int32_t         n_args;
    const int32_t*  args;          /* variable-length operand lists (PROBE keys)               */
    int32_t         sink_kind;
    int32_t         n_keys;        /* AGG: group keys; BUILD: join keys; MATERIALIZE: 0        */
    const rq_value* keys;
    int32_t         n_vals;        /* AGG: aggregates; BUILD: payload; MATERIALIZE: columns    */
    const rq_value* vals;
    int64_t         size_hint;     /* expected sink cardinality (RelOperator::getSize), 0 = ?  */
    int32_t         source_id2;    /* RQ_SRC_CROSS: the second materialized pipeline           */
    int32_t         reserved;
} rq_pipeline;
/* Output column order of a pipeline: keys first, then vals (aggregation.h:326). */

typedef struct {
    int32_t column;      /* column of the last pipeline's output                               */
    int32_t ascending;   /* 1 asc, 0 desc (qlib/sort.h:14)                                     */
} rq_order_key;

#define RQ_PLAN_SHARDED      1   /* the scanned fact table holds this rank's row range, the other
                                     tables are complete on every rank; partial aggregates are merged
                                     over NCCL                                                        */
#define RQ_PLAN_PARTITIONED  2   /* EVERY table holds this rank's row range (large join large): build
                                     and probe rows are shipped to the rank that owns hash(join key)
                                     (all-to-all: grouped ncclSend/ncclRecv), joined there, and the
                                     groups of the last aggregation are merged on the rank that owns
                                     hash(group key). The result is identical on every rank.          */

typedef struct {
    int32_t             n_tables;
    rq_table* const*    tables;
    int32_t             n_pipelines;
    const rq_pipeline*  pipelines;
    int32_t             n_order;       /* ORDER BY over the last pipeline (orderby.h:96-136)   */
    const rq_order_key* order;
    int64_t             limit;         /* -1 = none (Relation::applyLimit, dbdata.h:407)       */
    const char*         strpool;
    int64_t             strpool_bytes;
    int32_t             flags;
} rq_plan;

/* ---- result (replaces RelOperator::retrieveResult, RelOperator.h:182) -------------------- */
typedef struct {
    int32_t type;        /* RQ_I8 / RQ_I32 / RQ_I64 / RQ_STR                                   */
    int32_t width;       /* bytes per row                                                      */
    int32_t sql_type;    /* RQ_SQL_*                                                           */
    int32_t sql_width;   /* as rq_value.width                                                  */
    void*   data;        /* host memory, n_rows * width bytes, owned by the result             */
} rq_result_col;

typedef struct {
    int64_t        n_rows;
    int32_t        n_cols;
    rq_result_col* cols;
} rq_result;

/* Mirrors JitExecutionReport (JitContextFlounder.h:114-129): lower_ms ~ compilationTime,
 * kernel_ms ~ executionTime; the other phases are reported separately as north_star asks. */
typedef struct {
    double  lower_ms;        /* plan validation + program/slot assignment (host)               */
    double  h2d_ms;          /* host->device copies inside this call                           */
    double  kernel_ms;       /* CUDA-event time of all kernels of the plan                     */
    double  nccl_ms;         /* collective time (sharded plans)                                */
    double  d2h_ms;          /* result read-back                                               */
    double  scan_kernel_ms;  /* time of the table-scan pipeline kernels only (roofline)        */
    int32_t kernel_launches;
    int32_t host_syncs;      /* stream synchronisations the host waited for during this call     */
    double  fact_scan_ms;    /* the last table-scan kernel of the plan: the probe/aggregate
                                pipeline over the fact table (the roofline kernel)             */
} rq_timings;

int rq_plan_execute(const rq_plan* plan, rq_result** out, rq_timings* timings);
int rq_result_free(rq_result* r);

#ifdef __cplusplus
}
#endif
#endif /* RESQL_B200_H */
