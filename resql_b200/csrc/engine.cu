// resql_b200 engine: C ABI (include/resql_b200.h), device-resident columnar tables, lowering of
// the typed postfix programs to the accumulator-machine encoding, kernel orchestration.
//
// Replaces, on the reference side (Henning1/resql): JitContextFlounder::{compile,execute}
// (src/JitContextFlounder.h:410-487), the produceFlounder/consumeFlounder bodies of
// src/operators/*.h, qlib/hash.h and qlib/sort.h. No CPU fallback exists: every entry point fails
// with RQ_ERR_CUDA when no device is usable.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cstdarg>
#include <string>
#include <vector>
#include <map>
#include <set>
#include <memory>
#include <algorithm>
#include <chrono>
#include <functional>
#include <tuple>

#include "../../include/resql_b200.h"
#include "rq_internal.h"
#include "scan_kernel.cuh"
#include "sort_kernels.cuh"
#include "hash_kernels.cuh"
#include "exchange_kernels.cuh"
#include "dist.h"
#include "host_narrow.h"
#include "jit.h"
#include <thread>
#include <atomic>
#include <mutex>

using namespace rq;

// ------------------------------------------------------------------------------------------
// error handling
// ------------------------------------------------------------------------------------------
static std::string g_err;
static int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
struct RqError {
    int code;
    std::string msg;
};
[[noreturn]] static void raise(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    throw RqError{code, buf};
}
#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            raise(RQ_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),    \
                  __FILE__, __LINE__);                                                    \
    } while (0)

// ------------------------------------------------------------------------------------------
// engine state
// ------------------------------------------------------------------------------------------
// Storage layout. Tables the engine owns are stored TILE-MAJOR: the table is a sequence of pages of
// kTile (256) rows; a page holds the 256-row chunk of every fixed-width column back to back
// ([col0: 256 x w0][col1: 256 x w1]...). A warp tile of the scan kernel is exactly one page, so the
// chunks of all adjacent scanned columns arrive with ONE cp.async.bulk (every chunk is a multiple of
// 256 bytes: source, destination and size are always 16-byte aligned). String columns (accessed by
// address, never staged) stay plain arrays. Borrowed device columns and pipeline intermediates are
// plain arrays: one copy per column per tile.
struct DevColumn {
    int type = 0, width = 0;
    unsigned char* d = nullptr;     // plain array, or the column's chunk in page 0 of a tile-major table
    bool owned = true;
    int64_t tile_stride = 0;        // bytes from one tile's chunk to the next (plain: kTile * width)
    uint32_t page_off = 0;          // tile-major: offset of the chunk inside a page
    // exact value bounds over all rows, taken once at upload (the data of a table never changes
    // afterwards: the reference's tables are append-only and re-uploaded per version). They let the
    // lowering prove that a value fits in 32 bits and pick the narrow instruction forms.
    bool has_stats = false;
    int64_t vmin = 0, vmax = 0;
    bool sorted = false;            // values are non-decreasing over the rows (taken with the statistics): range
                                    // selections on this column restrict the scan to a row range
};
static uint64_t g_next_table_uid = 1;
struct rq_table {
    std::string name;
    uint64_t uid = g_next_table_uid++;      // identity of this upload (plan memos are keyed by it)
    int64_t n_rows = 0;       // host-known row count (-1: only on device)
    int64_t cap_rows = 0;     // allocated rows (multiple of kTileRows for owned tables)
    int64_t* d_n_rows = nullptr;
    bool borrowed = false;
    unsigned char* pax_base = nullptr;   // tile-major storage of the fixed-width columns (owned tables)
    size_t page_bytes = 0;
    std::vector<DevColumn> cols;
    // logical type info for intermediates (per column)
    std::vector<int> sql_type, sql_width;
    // nested-loops join source (RQ_SRC_CROSS): the pairs of two relation outputs, streamed by the scan
    // kernel and never materialized. `cols` aliases the columns of cross[0], then those of cross[1];
    // n_rows is the pair count; cross[cross_inner] is the relation iterated inside (scan_kernel.cuh)
    const rq_table* cross[2] = {nullptr, nullptr};
    int cross_inner = 1;
    ~rq_table() {
        for (auto& c : cols)
            if (c.owned && c.d) dfree(c.d);
        if (pax_base) dfree(pax_base);
        if (d_n_rows) dfree(d_n_rows);
    }
};

// knobs (rq_set_option): defaults are the production choices, tests force the rarely taken paths
struct Options {
    int stages = 0, warps = 0;            // override the shared-memory layout of the scan kernel (0 = automatic)
    int64_t split_min_rows = -1;          // two-pass probes: minimal table size (-1 = default 4 Mi rows)
    double split_frac = -1;               //                   maximal build/probe-domain ratio (-1 = default 0.3)
    bool prune_builds = true;             // restrict build sides to the probe key's value range
    bool topk = true;                     // ORDER BY ... LIMIT k through radix select
    bool direct_joins = true;             // direct-address join tables for dense unique integer keys
    bool group_joins = true;              // GROUP BY on the key of a direct-address join aggregates into its entries
    bool replay = true;                   // predicted host reads (engine_exec.inl "host reads of device values")
    bool graphs = true;                   // replayed plans are captured into CUDA graphs
    bool zone_skip = true;                // selections on sorted columns restrict the scan to a tile range
    int late_materialize = 1;             // 0 never, 1 where the early form cannot hold a materialize, 2 wherever it applies
    int sink_rounds = 1;                  // materialize values in rounds (engine_exec.inl "sink rounds"): 0 never, 1 where
                                          // the single sink cannot hold the values, 2 wherever it applies
    int in_lists = 1;                     // OR trees of equality tests against constants as one set test (engine_exec.inl
                                          // "IN lists"): 0 never, 1 lists of kInListMinInt / kInListMinStr values or more, 2 every list
    bool share_builds = true;             // sharded plans: replicated pure-scan builds are split over the ranks and all-reduced
    int64_t share_min_rows = 1 << 20;
    bool narrow = true;                   // host-buffer uploads send 8-byte columns over PCIe in the narrowest exact width
    int up_threads = 0;                   // host-buffer uploads: converting threads (0 = all cores of this rank's share)
    int up_chunk_krows = 512;             //                      rows per conversion / DMA chunk, in 1024 rows
    bool trace = false;                   // per-step wall-clock trace on stderr
    bool specialize = true;               // scan launches run a kernel compiled for their pipeline (jit.h)
};

struct Engine {
    bool init = false;
    Options opt;
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev[8];
    // scratch for the low-card aggregate path
    uint32_t* g_state = nullptr;
    int64_t* g_keys = nullptr;
    int64_t* g_acc = nullptr;
    uint8_t* g_kinds = nullptr;
    int32_t* flags = nullptr;   // FlagBlock (rq_internal.h), 64 bytes
    int32_t* h_flags = nullptr; // pinned
    unsigned char* pinned = nullptr;   // pinned scratch: host reads (4 KB) + ring of small uploads
    Dist dist;
    // host-buffer uploads: one converting thread per worker, each with its own stream and a
    // double-buffered pair of (pinned host, device) staging chunks (host_narrow.h)
    struct UpWorker { size_t cap = 0; double conv_ms = 0, wait_ms = 0; cudaStream_t s = nullptr; cudaEvent_t ev[2] = {nullptr, nullptr}; unsigned char* h[2] = {nullptr, nullptr}; unsigned char* d[2] = {nullptr, nullptr}; };
    std::vector<UpWorker> up;
    cudaEvent_t up_ready = nullptr;
};
static Engine E;

static int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
static constexpr int kSmemMax = 227 * 1024;

struct rq_table;
static void compute_stats(rq_table& t);
static void reset_plan_memos();

// ------------------------------------------------------------------------------------------
// lifecycle
// ------------------------------------------------------------------------------------------
extern "C" int rq_init(int device) {
    try {
        if (E.init) return RQ_OK;
        int n = 0;
        CK(cudaGetDeviceCount(&n));
        if (device < 0 || device >= n) return fail(RQ_ERR_CUDA, "rq_init: device %d of %d", device, n);
        CK(cudaSetDevice(device));
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10)
            return fail(RQ_ERR_CUDA, "rq_init: device %s is sm_%d%d, this engine is built for sm_100a",
                        prop.name, prop.major, prop.minor);
        E.device = device;
        E.sm_count = prop.multiProcessorCount;
        CK(cudaStreamCreateWithFlags(&E.stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&E.copy_stream, cudaStreamNonBlocking));
        alloc_stream() = E.stream;
        {   // keep freed blocks in the pool: hash tables and intermediates are recycled across queries
            cudaMemPool_t pool;
            CK(cudaDeviceGetDefaultMemPool(&pool, device));
            uint64_t keep = UINT64_MAX;
            CK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
        }
        for (auto& e : E.ev) CK(cudaEventCreate(&e));
        CK(dmalloc(&E.g_state, sizeof(uint32_t) * kGroupTableCap));
        CK(dmalloc(&E.g_keys, sizeof(int64_t) * kGroupTableCap));
        CK(dmalloc(&E.g_acc, sizeof(int64_t) * kGroupTableCap * kMaxAggs));
        CK(dmalloc(&E.g_kinds, kMaxAggs));
        CK(dmalloc(&E.flags, 64));
        CK(cudaMallocHost(&E.h_flags, 64));
        CK(cudaMallocHost(&E.pinned, 36864));
        // every kernel scan_kernel_for can return (some more than once)
        for (int gr : {0, 1, 4})
            for (bool cross : {false, true})
                for (bool late : {false, true})
                    for (bool rounds : {false, true})
                        CK(cudaFuncSetAttribute(scan_kernel_for(gr, cross, late, rounds), cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
        E.init = true;
        return RQ_OK;
    } catch (RqError& e) {
        return fail(e.code, "%s", e.msg.c_str());
    }
}

extern "C" int rq_shutdown(void) {
    if (!E.init) return RQ_OK;
    cudaDeviceSynchronize();
    // captured plans hold NCCL kernel nodes: ncclCommDestroy waits until every graph that refers to
    // the communicator is gone (measured: the 2-GPU test worker never left rq_shutdown), so the
    // memos - and with them the graph executables - go first
    reset_plan_memos();
    cudaDeviceSynchronize();
    dist_shutdown(E.dist);
    dfree(E.g_state); dfree(E.g_keys); dfree(E.g_acc); dfree(E.g_kinds);
    dfree(E.flags); cudaFreeHost(E.h_flags); cudaFreeHost(E.pinned);
    for (auto& w : E.up) {
        for (int b = 0; b < 2; b++) { if (w.h[b]) cudaFreeHost(w.h[b]); if (w.d[b]) cudaFree(w.d[b]); if (w.ev[b]) cudaEventDestroy(w.ev[b]); }
        if (w.s) cudaStreamDestroy(w.s);
    }
    if (E.up_ready) cudaEventDestroy(E.up_ready);
    reset_plan_memos();
    cudaStreamSynchronize(E.stream);
    for (auto& e : E.ev) cudaEventDestroy(e);
    cudaStreamDestroy(E.stream);
    cudaStreamDestroy(E.copy_stream);
    alloc_stream() = nullptr;
    E = Engine();
    return RQ_OK;
}

extern "C" const char* rq_last_error(void) { return g_err.c_str(); }

extern "C" int rq_set_option(const char* key, double value) {
    if (!key) return fail(RQ_ERR_INVALID, "rq_set_option: no key");
    const std::string k = key;
    Options& o = E.opt;
    if (k == "stages") o.stages = (int)value;
    else if (k == "warps") o.warps = (int)value;
    else if (k == "split_min_rows") o.split_min_rows = (int64_t)value;
    else if (k == "split_frac") o.split_frac = value;
    else if (k == "prune_builds") o.prune_builds = value != 0;
    else if (k == "topk") o.topk = value != 0;
    else if (k == "direct_joins") o.direct_joins = value != 0;
    else if (k == "group_joins") o.group_joins = value != 0;
    else if (k == "replay") o.replay = value != 0;
    else if (k == "graphs") o.graphs = value != 0;
    else if (k == "narrow") o.narrow = value != 0;
    else if (k == "zone_skip") o.zone_skip = value != 0;
    else if (k == "late_materialize") o.late_materialize = std::max(0, std::min((int)value, 2));
    else if (k == "sink_rounds") o.sink_rounds = std::max(0, std::min((int)value, 2));
    else if (k == "in_lists") o.in_lists = std::max(0, std::min((int)value, 2));
    else if (k == "share_builds") o.share_builds = value != 0;
    else if (k == "share_min_rows") o.share_min_rows = (int64_t)value;
    else if (k == "up_threads") o.up_threads = (int)value;
    else if (k == "up_chunk_krows") o.up_chunk_krows = std::max(1, std::min((int)value, 8192));
    else if (k == "trace") o.trace = value != 0;
    else if (k == "specialize") o.specialize = value != 0;
    else return fail(RQ_ERR_INVALID, "rq_set_option: unknown option '%s'", key);
    return RQ_OK;
}
extern "C" void* rq_stream(void) { return (void*)E.stream; }

extern "C" int rq_dist_unique_id(uint8_t out_id[128]) {
    std::string err;
    if (!dist_unique_id(out_id, err)) return fail(RQ_ERR_NCCL, "%s", err.c_str());
    return RQ_OK;
}
extern "C" int rq_dist_init(int rank, int world, const uint8_t id[128]) {
    if (!E.init) return fail(RQ_ERR_NOT_INIT, "rq_dist_init before rq_init");
    std::string err;
    if (!dist_init(E.dist, rank, world, id, err)) return fail(RQ_ERR_NCCL, "%s", err.c_str());
    // NCCL sets up its rings and peer-to-peer channels at the first use of every kind of operation
    // (seconds on 8 ranks: measured 7 s inside the first Q3). That belongs to joining the group, not to
    // the first query: one tiny collective of every kind the engine uses, and a send/receive with every
    // peer, are run here.
    if (world > 1) {
        Dist& D = E.dist;
        unsigned long long* buf = nullptr;
        if (cudaMalloc(&buf, sizeof(unsigned long long) * (size_t)(2 * world + 2)) == cudaSuccess) {
            cudaMemsetAsync(buf, 0, sizeof(unsigned long long) * (size_t)(2 * world + 2), E.stream);
            int rc = D.all_reduce(buf, buf, 1, 5, 0, D.comm, E.stream);
            if (rc == 0) rc = D.all_gather(buf + 2 * world, buf, 1, 5, D.comm, E.stream);
            if (rc == 0) rc = D.broadcast(buf, buf, 1, 5, 0, D.comm, E.stream);
            if (rc == 0) rc = D.group_start();
            for (int r = 0; r < world && rc == 0; r++) {
                if (r == rank) continue;
                rc = D.send(buf + world + r, 1, 5, r, D.comm, E.stream);
                if (rc == 0) rc = D.recv(buf + r, 1, 5, r, D.comm, E.stream);
            }
            if (rc == 0) rc = D.group_end();
            const cudaError_t ce = cudaStreamSynchronize(E.stream);
            cudaFree(buf);
            if (rc != 0 || ce != cudaSuccess) return fail(RQ_ERR_NCCL, "rq_dist_init: warm-up collectives failed");
        }
    }
    return RQ_OK;
}

// ------------------------------------------------------------------------------------------
// tables
// ------------------------------------------------------------------------------------------
static bool valid_col(int type, int width) {
    if (type == RQ_I8) return width == 1;
    if (type == RQ_I32) return width == 4;
    if (type == RQ_I64) return width == 8;
    if (type == RQ_STR) return width >= 2;
    return false;
}

// allocates the storage of an owned table (cap_rows must be set): fixed-width columns tile-major in
// one block, strings as plain arrays; everything behind n_rows is zero
template <typename FT, typename FW>
static void alloc_tile_major(rq_table& t, int n_cols, FT type_of, FW width_of) {
    size_t page = 0;
    for (int c = 0; c < n_cols; c++) {
        DevColumn dc;
        dc.type = type_of(c);
        dc.width = width_of(c);
        if (dc.type != RQ_STR) { dc.page_off = (uint32_t)page; page += (size_t)kTile * dc.width; dc.owned = false; }
        t.cols.push_back(dc);
    }
    t.page_bytes = page;
    const int64_t pages = t.cap_rows / kTile;
    if (page) {
        CK(dmalloc(&t.pax_base, (size_t)pages * page));
        // rows behind n_rows read as zero: clear from the page that holds row n_rows to the end
        const int64_t first = std::max<int64_t>(t.n_rows, 0) / kTile;
        CK(cudaMemsetAsync(t.pax_base + (size_t)first * page, 0, (size_t)(pages - first) * page, E.stream));
    }
    for (auto& dc : t.cols) {
        if (dc.type != RQ_STR) {
            dc.d = t.pax_base + dc.page_off;
            dc.tile_stride = (int64_t)page;
        } else {
            const size_t bytes = (size_t)t.cap_rows * dc.width;
            CK(dmalloc(&dc.d, bytes));
            dc.tile_stride = (int64_t)kTile * dc.width;
            const size_t used = (size_t)std::max<int64_t>(t.n_rows, 0) * dc.width;
            CK(cudaMemsetAsync(dc.d + used, 0, bytes - used, E.stream));
        }
    }
}

// ---- upload from host buffers with host-side narrowing (host_narrow.h) ------------------------------

static std::map<std::string, std::vector<int>> g_width_hint; // physical widths that held for a table name last time

// rows [row0, row0 + n) of a column, as they are, into their place in the table (row0 is a multiple of kTile)
static void copy_column_rows(rq_table& t, int c, const void* data, int64_t row0, int64_t n, cudaMemcpyKind kind, cudaStream_t st) {
    DevColumn& dc = t.cols[c];
    const unsigned char* src = (const unsigned char*)data + (size_t)row0 * dc.width;
    if (dc.type == RQ_STR) {
        if (n) CK(cudaMemcpyAsync(dc.d + (size_t)row0 * dc.width, src, (size_t)n * dc.width, kind, st));
        return;
    }
    // full pages with one pitched copy, the partial last page with a plain one
    unsigned char* dst = dc.d + (size_t)(row0 / kTile) * t.page_bytes;
    const size_t chunk = (size_t)kTile * dc.width;
    const int64_t full = n / kTile;
    if (full > 0) CK(cudaMemcpy2DAsync(dst, t.page_bytes, src, chunk, chunk, (size_t)full, kind, st));
    const size_t rest = (size_t)n * dc.width - (size_t)full * chunk;
    if (rest) CK(cudaMemcpyAsync(dst + (size_t)full * t.page_bytes, src + (size_t)full * chunk, rest, kind, st));
}
static void copy_column_plain(rq_table& t, int c, const void* data, int64_t n_rows, cudaMemcpyKind kind) {
    copy_column_rows(t, c, data, 0, n_rows, kind, E.stream);
}

// Returns the finished table, or null when no column can be narrowed (the caller takes the plain
// path). The table in HBM keeps the reference's widths (the scan kernel's operand forms and the
// roofline's algorithmic bytes are defined on them; with the present kernels Q1/Q6/Q3 are bound by
// instruction issue, not by HBM bytes, so narrower resident columns measured no gain - DESIGN.md):
// a chunk is widened again by rq_repack_col when it lands. The transfer width of every 8-byte column is guessed from a sample (or from the widths that
// held for the same table name before), the columns are converted chunk by chunk on all host cores
// while the exact value range is taken; a value that does not fit its guess widens the guess and the
// upload starts over (at most twice; data whose sample lies about its range is rare).
static std::unique_ptr<rq_table> upload_host_narrow(const char* name, int n_cols, const rq_column* cols, int64_t n_rows) {
    const int64_t kUpChunkRows = (int64_t)E.opt.up_chunk_krows * 1024;      // (a multiple of kTile)
    if (!E.opt.narrow || n_rows < 4 * kUpChunkRows) return nullptr;
    {   // Converting pays only while the host cores outrun the link: measured, one core converts about
        // 8 GB/s of 8-byte values and the link moves 52 GB/s, so with fewer than 7 cores for this rank
        // (several ranks share the host) the columns travel as they are - every rank has its own link.
        int hw = (int)std::thread::hardware_concurrency();
        const int share = E.opt.up_threads > 0 ? E.opt.up_threads : hw / std::max(1, E.dist.world);
        if (share < 7) return nullptr;
    }
    const std::string hint_key = std::string(name ? name : "") + "/" + std::to_string(n_cols);
    std::vector<int> gw(n_cols);
    {
        auto h = g_width_hint.find(hint_key);
        for (int c = 0; c < n_cols; c++) {
            gw[c] = cols[c].width;
            if (cols[c].type != RQ_I64 && cols[c].type != RQ_I32) continue;
            if (h != g_width_hint.end()) { gw[c] = h->second[c]; continue; }
            const int64_t step = std::max<int64_t>(1, n_rows / 4096);
            if (cols[c].type == RQ_I32) {           // 4-byte columns: one byte or as they are
                const int32_t* p = (const int32_t*)cols[c].data;
                int32_t lo = p[n_rows - 1], hi = lo;
                for (int64_t i = 0; i < n_rows; i += step) { lo = std::min(lo, p[i]); hi = std::max(hi, p[i]); }
                gw[c] = (lo >= 0 && hi <= 255) ? 1 : 4;
                continue;
            }
            const int64_t* p = (const int64_t*)cols[c].data;
            int64_t lo = p[n_rows - 1], hi = lo;
            for (int64_t i = 0; i < n_rows; i += step) { lo = std::min(lo, p[i]); hi = std::max(hi, p[i]); }
            gw[c] = (lo >= 0 && hi <= 255) ? 1 : (lo >= INT32_MIN && hi <= INT32_MAX) ? 4 : 8;
        }
    }
    const auto t_begin = std::chrono::steady_clock::now();
    for (int attempt = 0; attempt < 3; attempt++) {
        std::vector<int> ncols;
        auto narrowed = [&](int c) { return (cols[c].type == RQ_I64 || cols[c].type == RQ_I32) && gw[c] != cols[c].width; };
        for (int c = 0; c < n_cols; c++) if (narrowed(c)) ncols.push_back(c);
        if (ncols.empty()) { g_width_hint[hint_key] = gw; return nullptr; }
        std::unique_ptr<rq_table> t(new rq_table());
        t->name = name ? name : "";
        t->n_rows = n_rows;
        t->cap_rows = round_up(std::max<int64_t>(n_rows, 1), kPadRows);
        alloc_tile_major(*t, n_cols, [&](int c) { return cols[c].type; }, [&](int c) { return cols[c].width; });
        if (!E.up_ready) CK(cudaEventCreateWithFlags(&E.up_ready, cudaEventDisableTiming));
        CK(cudaEventRecord(E.up_ready, E.stream));            // storage allocated and cleared
        // columns that travel as they are: queued first, the link is busy while the host converts
        // Work items are (row chunk, column) pairs in chunk-major order: a narrowed column is converted
        // into a staging buffer and copied from there, any other column is copied as it is - from the
        // same queue, so that the copy engine always has both kinds of chunks to move while the host
        // converts (one huge copy per direct column in front would keep the engine to itself: measured,
        // the converted chunks then wait and nothing overlaps).
        std::vector<int> icols;
        for (int c = 0; c < n_cols; c++) icols.push_back(c);
        const int64_t chunks = (n_rows + kUpChunkRows - 1) / kUpChunkRows;
        const int64_t n_items = chunks * (int64_t)icols.size();
        int T = (int)std::thread::hardware_concurrency();
        T = std::max(2, std::min(T / std::max(1, E.dist.world), 32));
        if (E.opt.up_threads > 0) T = std::min(E.opt.up_threads, 64);
        T = (int)std::min<int64_t>(T, n_items);
        for (auto& w : E.up)                        // chunk size raised since the buffers were made
            if (w.cap < (size_t)kUpChunkRows * 4) {
                for (int b = 0; b < 2; b++) {
                    CK(cudaFreeHost(w.h[b])); CK(cudaFree(w.d[b]));
                    CK(cudaMallocHost(&w.h[b], (size_t)kUpChunkRows * 4));
                    CK(cudaMalloc(&w.d[b], (size_t)kUpChunkRows * 4));
                }
                w.cap = (size_t)kUpChunkRows * 4;
            }
        while ((int)E.up.size() < T) {
            Engine::UpWorker w;
            CK(cudaStreamCreateWithFlags(&w.s, cudaStreamNonBlocking));
            for (int b = 0; b < 2; b++) {
                CK(cudaEventCreateWithFlags(&w.ev[b], cudaEventDisableTiming));
                CK(cudaMallocHost(&w.h[b], (size_t)kUpChunkRows * 4));
                CK(cudaMalloc(&w.d[b], (size_t)kUpChunkRows * 4));
                w.cap = (size_t)kUpChunkRows * 4;
            }
            E.up.push_back(w);
        }
        std::atomic<int64_t> next{0};
        std::atomic<int> bad_col{-1};
        std::atomic<int> cuda_err{0};
        std::mutex mu;
        std::vector<int64_t> lo(n_cols, INT64_MAX), hi(n_cols, INT64_MIN);
        auto work = [&](int tid) {
            Engine::UpWorker& w = E.up[tid];
            if (cudaSetDevice(E.device) != cudaSuccess || cudaStreamWaitEvent(w.s, E.up_ready, 0) != cudaSuccess) { cuda_err = 1; return; }
            std::vector<int64_t> tlo(n_cols, INT64_MAX), thi(n_cols, INT64_MIN);
            int b = 0;
            bool used[2] = {false, false};
            for (;;) {
                const int64_t it = next.fetch_add(1);
                if (it >= n_items || bad_col.load() >= 0 || cuda_err.load()) break;
                // chunk-major order: the chunks of all narrowed columns of a row range are converted together
                const int c = icols[(size_t)(it % (int64_t)icols.size())];
                const int64_t row0 = (it / (int64_t)icols.size()) * kUpChunkRows;
                const int64_t n = std::min<int64_t>(kUpChunkRows, n_rows - row0);
                const int w8 = gw[c];
                if (!narrowed(c)) {
                    try { copy_column_rows(*t, c, cols[c].data, row0, n, cudaMemcpyHostToDevice, w.s); }
                    catch (RqError&) { cuda_err = 1; break; }
                    continue;
                }
                const auto t0 = std::chrono::steady_clock::now();
                if (used[b] && cudaEventSynchronize(w.ev[b]) != cudaSuccess) { cuda_err = 1; break; }
                const auto t1 = std::chrono::steady_clock::now();
                const bool fits = cols[c].type == RQ_I32
                                      ? hostnarrow::convert_chunk32((const int32_t*)cols[c].data + row0, w.h[b], (size_t)n, &tlo[c], &thi[c])
                                      : hostnarrow::convert_chunk((const int64_t*)cols[c].data + row0, w.h[b], (size_t)n, w8, &tlo[c], &thi[c]);
                if (!fits) {
                    bad_col = c;
                    break;
                }
                w.wait_ms += std::chrono::duration<double, std::milli>(t1 - t0).count();
                w.conv_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count();
                const DevColumn& dc = t->cols[c];
                const int grid = (int)std::min<int64_t>((n + 255) / 256, 1024);
                bool ok = cudaMemcpyAsync(w.d[b], w.h[b], (size_t)n * w8, cudaMemcpyHostToDevice, w.s) == cudaSuccess;
                rq_repack_col<<<grid, 256, 0, w.s>>>(w.d[b], w8, dc.d + (size_t)(row0 / kTile) * dc.tile_stride, dc.width, dc.tile_stride, n);
                ok = ok && cudaGetLastError() == cudaSuccess && cudaEventRecord(w.ev[b], w.s) == cudaSuccess;
                if (!ok) { cuda_err = 1; break; }
                used[b] = true;
                b ^= 1;
            }
            if (cudaStreamSynchronize(w.s) != cudaSuccess) cuda_err = 1;
            std::lock_guard<std::mutex> g(mu);
            for (int c = 0; c < n_cols; c++) { lo[c] = std::min(lo[c], tlo[c]); hi[c] = std::max(hi[c], thi[c]); }
        };
        for (auto& w : E.up) { w.conv_ms = 0; w.wait_ms = 0; }
        std::vector<std::thread> th;
        for (int i = 1; i < T; i++) th.emplace_back(work, i);
        work(0);
        for (auto& x : th) x.join();
        if (cuda_err.load()) raise(RQ_ERR_CUDA, "rq_table_upload: a staging copy failed: %s", cudaGetErrorString(cudaGetLastError()));
        if (bad_col.load() >= 0) {
            // the sample lied: widen that column's guess and start over
            const int c = bad_col.load();
            gw[c] = cols[c].type == RQ_I32 ? 4 : (gw[c] == 1 ? 4 : 8);
            CK(cudaStreamSynchronize(E.stream));
            continue;
        }
        for (int c : ncols) { t->cols[c].has_stats = true; t->cols[c].vmin = lo[c]; t->cols[c].vmax = hi[c]; }
        g_width_hint[hint_key] = gw;
        if (E.opt.trace) {
            const double conv_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
            CK(cudaStreamSynchronize(E.stream));
            const double all_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
            size_t wire = 0, logical = 0;
            for (int c = 0; c < n_cols; c++) { wire += (size_t)n_rows * gw[c]; logical += (size_t)n_rows * cols[c].width; }
            double cv = 0, wt = 0;
            for (int i = 0; i < T; i++) { cv += E.up[i].conv_ms; wt += E.up[i].wait_ms; }
            fprintf(stderr, "[rq] upload %s: %lld rows, %d of %d columns narrowed on %d host threads (attempt %d): %.1f MB on the wire for %.1f MB, "
                            "conversion done after %.1f ms (per thread: %.1f ms converting, %.1f ms waiting for its staging buffers), "
                            "all copies after %.1f ms (%.1f GB/s of table bytes)\n",
                    t->name.c_str(), (long long)n_rows, (int)ncols.size(), n_cols, T, attempt, wire / 1e6, logical / 1e6, conv_ms, cv / T, wt / T,
                    all_ms, logical / 1e6 / all_ms);
        }
        return t;
    }
    return nullptr;
}

// debug aid (no GPU needed, not part of the public ABI): the host-side conversion of one chunk, so that the
// CPU-only tests can check fit detection and value ranges (tests/test_host_narrow.py)
extern "C" int rq_debug_convert_chunk(const int64_t* in, int64_t n, int32_t width, uint8_t* out, int64_t* lo, int64_t* hi) {
    if (!in || !out || !lo || !hi || n < 0 || (width != 1 && width != 4 && width != -1)) return -1;
    *lo = INT64_MAX; *hi = INT64_MIN;
    if (width == -1) return hostnarrow::convert_chunk32((const int32_t*)in, out, (size_t)n, lo, hi) ? 1 : 0;    // int32 source -> bytes
    return hostnarrow::convert_chunk(in, out, (size_t)n, width, lo, hi) ? 1 : 0;
}

extern "C" int rq_table_upload(const char* name, int32_t n_cols, const rq_column* cols,
                               int64_t n_rows, int32_t flags, rq_table** out) {
    if (!E.init) return fail(RQ_ERR_NOT_INIT, "rq_table_upload before rq_init");
    if (!out || n_cols <= 0 || !cols || n_rows < 0) return fail(RQ_ERR_INVALID, "rq_table_upload: bad arguments");
    std::unique_ptr<rq_table> t(new rq_table());
    try {
        t->name = name ? name : "";
        t->n_rows = n_rows;
        const bool dev = flags & RQ_DEVICE_PTR;
        const bool borrow = dev && (flags & RQ_BORROW);
        t->borrowed = borrow;
        t->cap_rows = borrow ? n_rows : round_up(std::max<int64_t>(n_rows, 1), kPadRows);
        for (int c = 0; c < n_cols; c++)
            if (!valid_col(cols[c].type, cols[c].width))
                raise(RQ_ERR_INVALID, "rq_table_upload: column %d has bad type/width %d/%d", c, cols[c].type, cols[c].width);
        if (!dev) {
            std::unique_ptr<rq_table> nt = upload_host_narrow(name, n_cols, cols, n_rows);
            if (nt) {
                compute_stats(*nt);
                CK(cudaStreamSynchronize(E.stream));
                *out = nt.release();
                return RQ_OK;
            }
        }
        if (!borrow) alloc_tile_major(*t, n_cols, [&](int c) { return cols[c].type; }, [&](int c) { return cols[c].width; });
        const cudaMemcpyKind kind = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        for (int c = 0; c < n_cols; c++) {
            if (borrow) {
                DevColumn dc;
                dc.type = cols[c].type;
                dc.width = cols[c].width;
                if (((uintptr_t)cols[c].data & 15) != 0)
                    raise(RQ_ERR_INVALID, "rq_table_upload: borrowed column %d is not 16-byte aligned", c);
                dc.d = (unsigned char*)cols[c].data;
                dc.owned = false;
                dc.tile_stride = (int64_t)kTile * dc.width;
                t->cols.push_back(dc);
                continue;
            }
            copy_column_plain(*t, c, cols[c].data, n_rows, kind);
        }
        compute_stats(*t);
        CK(cudaStreamSynchronize(E.stream));
    } catch (RqError& e) {
        return fail(e.code, "%s", e.msg.c_str());
    }
    *out = t.release();
    return RQ_OK;
}

extern "C" int rq_table_upload_rows(const char* name, int32_t n_cols, const int32_t* types,
                                    const int32_t* widths, const int32_t* offsets,
                                    int32_t tuple_size, int32_t n_blocks,
                                    const uint8_t* const* blocks, const size_t* block_bytes,
                                    rq_table** out) {
    if (!E.init) return fail(RQ_ERR_NOT_INIT, "rq_table_upload_rows before rq_init");
    if (!out || n_cols <= 0 || tuple_size <= 0 || n_blocks < 0) return fail(RQ_ERR_INVALID, "rq_table_upload_rows: bad arguments");
    std::unique_ptr<rq_table> t(new rq_table());
    unsigned char* d_rows[2] = {nullptr, nullptr};
    try {
        int64_t n_rows = 0;
        size_t max_block = 0;
        for (int b = 0; b < n_blocks; b++) {
            if (block_bytes[b] % tuple_size) raise(RQ_ERR_INVALID, "block %d holds a partial tuple", b);
            n_rows += block_bytes[b] / tuple_size;
            max_block = std::max(max_block, block_bytes[b]);
        }
        t->name = name ? name : "";
        t->n_rows = n_rows;
        t->cap_rows = round_up(std::max<int64_t>(n_rows, 1), kPadRows);
        for (int c = 0; c < n_cols; c++)
            if (!valid_col(types[c], widths[c]) || offsets[c] < 0 || offsets[c] + widths[c] > tuple_size)
                raise(RQ_ERR_INVALID, "rq_table_upload_rows: column %d bad type/width/offset", c);
        alloc_tile_major(*t, n_cols, [&](int c) { return types[c]; }, [&](int c) { return widths[c]; });
        if (max_block) {
            CK(dmalloc(&d_rows[0], max_block));
            CK(dmalloc(&d_rows[1], max_block));
        }
        int64_t row0 = 0;
        cudaEvent_t done[2];
        CK(cudaEventCreate(&done[0]));
        CK(cudaEventCreate(&done[1]));
        for (int b = 0; b < n_blocks; b++) {
            const int s = b & 1;
            const int64_t n = block_bytes[b] / tuple_size;
            if (n == 0) continue;
            if (b >= 2) CK(cudaEventSynchronize(done[s]));
            CK(cudaMemcpyAsync(d_rows[s], blocks[b], block_bytes[b], cudaMemcpyHostToDevice, E.stream));
            for (int c = 0; c < n_cols; c++) {
                rq_transpose_rows<<<(unsigned)((n + 255) / 256), 256, 0, E.stream>>>(
                    d_rows[s], n, tuple_size, offsets[c], widths[c], t->cols[c].d, t->cols[c].tile_stride, row0);
            }
            CK(cudaEventRecord(done[s], E.stream));
            row0 += n;
        }
        compute_stats(*t);
        CK(cudaStreamSynchronize(E.stream));
        CK(cudaGetLastError());
        cudaEventDestroy(done[0]);
        cudaEventDestroy(done[1]);
        dfree(d_rows[0]);
        dfree(d_rows[1]);
    } catch (RqError& e) {
        dfree(d_rows[0]);
        dfree(d_rows[1]);
        return fail(e.code, "%s", e.msg.c_str());
    }
    *out = t.release();
    return RQ_OK;
}

extern "C" int rq_table_alloc(const char* name, int32_t n_cols, const int32_t* types, const int32_t* widths,
                              int64_t n_rows, rq_table** out) {
    if (!E.init) return fail(RQ_ERR_NOT_INIT, "rq_table_alloc before rq_init");
    if (!out || n_cols <= 0 || !types || !widths || n_rows < 0) return fail(RQ_ERR_INVALID, "rq_table_alloc: bad arguments");
    std::unique_ptr<rq_table> t(new rq_table());
    try {
        t->name = name ? name : "";
        t->n_rows = n_rows;
        t->cap_rows = round_up(std::max<int64_t>(n_rows, 1), kPadRows);
        for (int c = 0; c < n_cols; c++)
            if (!valid_col(types[c], widths[c])) raise(RQ_ERR_INVALID, "rq_table_alloc: column %d has bad type/width %d/%d", c, types[c], widths[c]);
        alloc_tile_major(*t, n_cols, [&](int c) { return types[c]; }, [&](int c) { return widths[c]; });
        CK(cudaStreamSynchronize(E.stream));
    } catch (RqError& e) {
        return fail(e.code, "%s", e.msg.c_str());
    }
    *out = t.release();
    return RQ_OK;
}

extern "C" int rq_table_broadcast(rq_table* t, int32_t root) {
    if (!E.init) return fail(RQ_ERR_NOT_INIT, "rq_table_broadcast before rq_init");
    if (!t || t->borrowed) return fail(RQ_ERR_INVALID, "rq_table_broadcast: needs a table the engine owns");
    Dist& D = E.dist;
    if (!D.comm || D.world <= 1) return RQ_OK;
    if (root < 0 || root >= D.world) return fail(RQ_ERR_INVALID, "rq_table_broadcast: root %d of %d ranks", root, D.world);
    try {
        // the layout is a function of the schema and the row count, which all ranks passed alike: a
        // rank that disagrees would make the collective hang or scribble, so the shapes are compared first
        int64_t shape[4] = {t->n_rows, (int64_t)t->cols.size(), (int64_t)t->page_bytes, t->cap_rows};
        for (auto& c : t->cols) shape[2] = shape[2] * 131 + c.width * 7 + c.type;
        int64_t* d_shape = nullptr;
        CK(dmalloc(&d_shape, sizeof(shape) * (size_t)(D.world + 1)));
        CK(cudaMemcpyAsync(d_shape + 4 * D.world, shape, sizeof(shape), cudaMemcpyHostToDevice, E.stream));
        int rc = D.all_gather(d_shape + 4 * D.world, d_shape, 4, 4 /* ncclInt64 */, D.comm, E.stream);
        if (rc != 0) raise(RQ_ERR_NCCL, "ncclAllGather(table shape) failed: %s", D.get_error_string ? D.get_error_string(rc) : "?");
        std::vector<int64_t> all(4 * (size_t)D.world);
        CK(cudaMemcpyAsync(all.data(), d_shape, all.size() * 8, cudaMemcpyDeviceToHost, E.stream));
        CK(cudaStreamSynchronize(E.stream));
        dfree(d_shape);
        for (int r = 0; r < D.world; r++)
            if (memcmp(&all[4 * (size_t)r], shape, sizeof(shape)) != 0)
                raise(RQ_ERR_INVALID, "rq_table_broadcast: rank %d holds a table of another shape (%lld rows) than rank %d (%lld rows)",
                      r, (long long)all[4 * (size_t)r], D.rank, (long long)t->n_rows);
        if (t->pax_base) {
            const size_t bytes = (size_t)(t->cap_rows / kTile) * t->page_bytes;
            rc = D.broadcast(t->pax_base, t->pax_base, bytes, 0 /* ncclInt8 */, root, D.comm, E.stream);
            if (rc != 0) raise(RQ_ERR_NCCL, "ncclBroadcast(table pages) failed: %s", D.get_error_string ? D.get_error_string(rc) : "?");
        }
        for (auto& c : t->cols) {
            if (c.type != RQ_STR) continue;
            rc = D.broadcast(c.d, c.d, (size_t)t->cap_rows * c.width, 0, root, D.comm, E.stream);
            if (rc != 0) raise(RQ_ERR_NCCL, "ncclBroadcast(string column) failed: %s", D.get_error_string ? D.get_error_string(rc) : "?");
        }
        for (auto& c : t->cols) c.has_stats = false;
        compute_stats(*t);
        CK(cudaStreamSynchronize(E.stream));
        t->uid = g_next_table_uid++;          // new contents: plans recorded against the old ones do not apply
    } catch (RqError& e) {
        return fail(e.code, "%s", e.msg.c_str());
    }
    return RQ_OK;
}

// min / max and sortedness of every integer column (passes over the resident data, on the engine stream)
static void compute_stats(rq_table& t) {
    if (t.n_rows <= 0) return;
    std::vector<int> idx;
    for (size_t c = 0; c < t.cols.size(); c++)
        if (t.cols[c].type != RQ_STR) idx.push_back((int)c);
    if (idx.empty()) return;
    // per column: [min][max][sorted flag (int32) + pad]
    int64_t* d = nullptr;
    CK(dmalloc(&d, idx.size() * 24));
    std::vector<int64_t> h(idx.size() * 3);
    for (size_t k = 0; k < idx.size(); k++) { h[3 * k] = INT64_MAX; h[3 * k + 1] = INT64_MIN; h[3 * k + 2] = 1; }
    CK(cudaMemcpyAsync(d, h.data(), h.size() * 8, cudaMemcpyHostToDevice, E.stream));
    for (size_t k = 0; k < idx.size(); k++) {
        const DevColumn& dc = t.cols[idx[k]];
        const int grid = (int)std::min<int64_t>((t.n_rows + 256 * 16 - 1) / (256 * 16), (int64_t)E.sm_count * 8);
        if (!dc.has_stats)            // (host-converted columns bring their range)
            rq_col_minmax<<<std::max(grid, 1), 256, 0, E.stream>>>(dc.d, dc.width, dc.tile_stride, t.n_rows, d + 3 * k);
        rq_col_sorted<<<std::max(grid, 1), 256, 0, E.stream>>>(dc.d, dc.width, dc.tile_stride, t.n_rows, (int32_t*)(d + 3 * k + 2));
    }
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h.data(), d, h.size() * 8, cudaMemcpyDeviceToHost, E.stream));
    CK(cudaStreamSynchronize(E.stream));
    dfree(d);
    for (size_t k = 0; k < idx.size(); k++) {
        DevColumn& dc = t.cols[idx[k]];
        if (!dc.has_stats) { dc.has_stats = true; dc.vmin = h[3 * k]; dc.vmax = h[3 * k + 1]; }
        dc.sorted = (int32_t)(h[3 * k + 2] & 0xffffffff) != 0;
    }
}

extern "C" int64_t rq_table_rows(const rq_table* t) { return t ? t->n_rows : -1; }
extern "C" int rq_table_free(rq_table* t) {
    if (E.init) cudaStreamSynchronize(E.stream);
    delete t;
    return RQ_OK;
}

// ------------------------------------------------------------------------------------------
// lowering: ABI postfix program -> accumulator-machine instructions (no code generation)
// ------------------------------------------------------------------------------------------
namespace {

struct PipeOut {                    // what a finished pipeline left on the device
    std::unique_ptr<rq_table> table;   // AGG / MATERIALIZE output (int64 columns)
    std::unique_ptr<HashTableDev> ht;  // BUILD output
    std::vector<int> payload_sql_type, payload_sql_width;
    std::vector<uint8_t> pay_word;     // BUILD: payload index (as in the plan) -> entry word, 0xff = not stored
    bool gj = false;                   // BUILD: direct-address entries carry the accumulators of a groupjoin,
    std::vector<int> gj_kind;          //        of these aggregate kinds, from entry word gj_word on
    uint32_t gj_word = 0;
    std::vector<void*> owned;          // device buffers the relation's string addresses point into
    ~PipeOut() { for (void* p : owned) dfree(p); }
    PipeOut() = default;
    PipeOut(PipeOut&&) = default;
    PipeOut& operator=(PipeOut&&) = default;
};

bool is_leaf(int op) { return op == RQ_OP_COL || op == RQ_OP_CONST || op == RQ_OP_CONST_STR; }
// Nodes only late materialization builds (never accepted from the ABI, run_pipeline checks): the
// absolute row (pair) index of the tuple, and PAYLOAD with b = kPayloadEntry, the reference of the
// probe's matched entry (scan kernel variant LATE).
constexpr int kOpRowId = 1000;
constexpr int kPayloadEntry = -1;
// Node only simplify_pipeline builds (never accepted from the ABI either): a = value, imm = key of a
// constant set in g_inlists; 1 when the value is in the set (an IN list, engine_exec.inl "IN lists").
constexpr int kOpInSet = 1001;
bool is_binary(int op) {
    switch (op) {
        case RQ_OP_ADD: case RQ_OP_SUB: case RQ_OP_MUL: case RQ_OP_DIV: case RQ_OP_AND: case RQ_OP_OR:
        case RQ_OP_LT: case RQ_OP_LE: case RQ_OP_GT: case RQ_OP_GE: case RQ_OP_EQ: case RQ_OP_NEQ:
        case RQ_OP_EQ_CHAR: case RQ_OP_EQ_VARCHAR: case RQ_OP_NEQ_CHAR: case RQ_OP_NEQ_VARCHAR:
        case RQ_OP_LIKE:
            return true;
        default:
            return false;
    }
}
// device opcode of a binary ABI op
uint8_t dop_left(int op) {
    switch (op) {
        case RQ_OP_ADD: return D_ADD; case RQ_OP_SUB: return D_SUB; case RQ_OP_MUL: return D_MUL;
        case RQ_OP_DIV: return D_DIV; case RQ_OP_AND: return D_AND; case RQ_OP_OR: return D_OR;
        case RQ_OP_LT: return D_LT; case RQ_OP_LE: return D_LE; case RQ_OP_GT: return D_GT;
        case RQ_OP_GE: return D_GE; case RQ_OP_EQ: return D_EQ; case RQ_OP_NEQ: return D_NE;
        case RQ_OP_EQ_CHAR: return D_EQC; case RQ_OP_EQ_VARCHAR: return D_EQV;
        case RQ_OP_NEQ_CHAR: return D_NEC; case RQ_OP_NEQ_VARCHAR: return D_NEV;
        case RQ_OP_LIKE: return D_LIKE;
    }
    return 0;
}
// selection-fused compare: column CMP constant (constant on the right / on the left)
uint8_t fcmp_left(int op) {
    switch (op) {
        case RQ_OP_LT: return D_LT; case RQ_OP_LE: return D_LE; case RQ_OP_GT: return D_GT;
        case RQ_OP_GE: return D_GE; case RQ_OP_EQ: return D_EQ; case RQ_OP_NEQ: return D_NE;
    }
    return 0;
}
uint8_t fcmp_right(int op) {
    switch (op) {
        case RQ_OP_LT: return D_GT; case RQ_OP_LE: return D_GE; case RQ_OP_GT: return D_LT;
        case RQ_OP_GE: return D_LE; case RQ_OP_EQ: return D_EQ; case RQ_OP_NEQ: return D_NE;
    }
    return 0;
}

struct HOpnd {           // host-level operand of a unit / value reference of a sink
    uint8_t kind = S_NONE;   // DSrc
    uint16_t idx = 0;        // staged column / slot / string column (sinks: imm-table index)
    int64_t imm = 0;
    uint8_t u32 = 0;         // value proven to lie in [0, 2^32)
    int64_t lo = INT64_MIN, hi = INT64_MAX;   // sinks: value bounds (group-key packing)
};
typedef HOpnd HRef;

enum HOp : uint8_t { H_FCMP = 1, H_BIN = 2, H_MULI = 3, H_SEL = 4, H_PROBE = 5, H_FRANGE = 6, H_INSET = 7 };

// One unit of the host-level program (what tests/vm_model.py executes):
//   H_FCMP  valid &= (x GOP imm)                      gop in D_LT..D_NE, x a column
//   H_BIN   t = x GOP y  (GOP = D_LD: t = x)
//   H_MULI  t = (x GOP imm) * y                       gop in D_ADD / D_SUB / D_RSUB
//   H_SEL   t = (x & 0xff) ? y : z
//   H_PROBE hash-join probe number aux
//   H_FRANGE valid &= (imm <= x <= imm + imm2)         two H_FCMP on one column fused
//   H_INSET t = (x in the constant set at device address imm)   (modelled by tests/vm_model_inset.py)
// then  slot[dst] = t  if dst >= 0, and  valid &= (t & 0xff) != 0  if filt.
struct HUnit {
    uint8_t op = 0, gop = 0;
    HOpnd x, y, z;
    int64_t imm = 0, imm2 = 0;
    int dst = -1;
    bool filt = false;
    int aux = 0;
    bool n32 = false;        // both multiplication factors proven to lie in [0, 2^32)
    int round = 0;           // sink rounds: 0 the prefix, k + 1 round k
};

struct Lowerer {
    const rq_plan& plan;
    const rq_pipeline& pl;
    const rq_table& src;
    const std::vector<PipeOut>& outs;
    const char* d_strpool;
    KParams& P;

    int n;
    std::vector<HUnit> prog;
    std::vector<HRef> hkey, hout;
    HRef hagg_src[kMaxAggs];
    HRef hprobe_key[kMaxProbes][kMaxKeys];
    int n_slots = 0;
    int row_slot = -1;                // slot of the kOpRowId node (late materialization)
    // sink rounds (engine_exec.inl "sink rounds"): round k stores values [round_val_end[k - 1],
    // round_val_end[k]); empty: one sink after the whole program
    std::vector<int> round_val_end;
    int cur_round = 0;                // the round of the units emitted now
    bool out_of_slots = false;        // the lowering failed for want of a value slot
    bool allow_rounds = true;         // the pipeline may take the round form

    std::vector<int> uses;            // consumers per node
    std::vector<int> last_use;        // last consuming node index (n = sink)
    std::vector<char> sink_ref;       // referenced by the sink or a probe key
    std::vector<int> slot;            // assigned slot or -1
    std::vector<HOpnd> leaf_op;       // operand descriptor of leaves
    std::vector<int> staged_of_col;   // source column -> staged index / str index
    std::vector<int> free_slots;
    std::vector<char> fused;          // node produces no unit of its own (folded into a consumer)
    std::vector<__int128> vlo, vhi;   // value bounds per node (full int64 range when unknown)
    int n_imm = 0;

    Lowerer(const rq_plan& plan, const rq_pipeline& pl, const rq_table& src,
            const std::vector<PipeOut>& outs, const char* d_strpool, KParams& P)
        : plan(plan), pl(pl), src(src), outs(outs), d_strpool(d_strpool), P(P), n(pl.n_nodes) {}

    void check_ref(int i, int ref) {
        if (ref < 0 || ref >= i) raise(RQ_ERR_INVALID, "node %d refers to node %d (must be an earlier node)", i, ref);
    }

    HUnit& emit(uint8_t op, uint8_t gop) {
        if ((int)prog.size() >= kMaxInsn) raise(RQ_ERR_UNSUPPORTED, "program longer than %d units", kMaxInsn);
        HUnit u;
        u.op = op; u.gop = gop;
        u.round = cur_round;
        prog.push_back(u);
        return prog.back();
    }

    HOpnd operand_of(int node) {
        if (is_leaf(pl.nodes[node].op)) return leaf_op[node];
        if (slot[node] < 0) raise(RQ_ERR_INVALID, "internal: node %d has no slot", node);
        HOpnd o; o.kind = S_SLOT; o.idx = (uint16_t)slot[node];
        return o;
    }
    HRef href_of(int node) {
        HRef v = operand_of(node);
        v.u32 = is_u32(node) ? 1 : 0;
        v.lo = (int64_t)vlo[node]; v.hi = (int64_t)vhi[node];
        if (v.kind == S_IMM) {
            if (n_imm >= kMaxImm) raise(RQ_ERR_UNSUPPORTED, "too many constants in sink");
            P.imm[n_imm] = v.imm;
            v.idx = (uint16_t)n_imm++;
        }
        return v;
    }
    int imm_index(int64_t v) {
        if (n_imm >= kMaxImm) raise(RQ_ERR_UNSUPPORTED, "too many constants");
        P.imm[n_imm] = v;
        return n_imm++;
    }

    int alloc_slot() {
        if (!free_slots.empty()) { int s = free_slots.back(); free_slots.pop_back(); return s; }
        if (n_slots >= kMaxSlots) out_of_slots = true;
        if (n_slots >= kMaxSlots) raise(RQ_ERR_UNSUPPORTED, "expression needs more than %d live temporaries", kMaxSlots);
        return n_slots++;
    }
    void release_dead(int at) {   // free slots of nodes whose last use is `at`
        for (int i = 0; i < n; i++)
            if (slot[i] >= 0 && last_use[i] == at) { free_slots.push_back(slot[i]); slot[i] = -2 - slot[i]; }
    }

    // back to the state before prepare(), keeping round_val_end (a second lowering of the pipeline)
    void reset() {
        prog.clear(); hkey.clear(); hout.clear();
        for (HRef& h : hagg_src) h = HRef();
        for (auto& k : hprobe_key) for (HRef& h : k) h = HRef();
        n_slots = 0; row_slot = -1; cur_round = 0; out_of_slots = false;
        free_slots.clear();
        n_imm = 0;
    }

    void prepare() {
        uses.assign(n, 0); last_use.assign(n, -1); sink_ref.assign(n, 0); slot.assign(n, -1);
        leaf_op.assign(n, HOpnd()); fused.assign(n, 0);
        staged_of_col.assign(src.cols.size(), -1);
        auto use = [&](int i, int ref) { check_ref(i, ref); uses[ref]++; last_use[ref] = std::max(last_use[ref], i); };
        for (int i = 0; i < n; i++) {
            const rq_node& nd = pl.nodes[i];
            switch (nd.op) {
                case RQ_OP_COL: {
                    if (nd.a < 0 || nd.a >= (int)src.cols.size()) raise(RQ_ERR_INVALID, "node %d: column %d out of range", i, nd.a);
                    const DevColumn& dc = src.cols[nd.a];
                    HOpnd o;
                    if (dc.type == RQ_STR) {
                        if (staged_of_col[nd.a] < 0) {
                            if (P.n_strcols >= kMaxStrCols) raise(RQ_ERR_UNSUPPORTED, "too many string columns");
                            P.str_ptr[P.n_strcols] = dc.d; P.str_w[P.n_strcols] = dc.width;
                            staged_of_col[nd.a] = P.n_strcols++;
                        }
                        o.kind = S_STR;
                    } else {
                        if (staged_of_col[nd.a] < 0) {
                            if (P.n_cols >= kMaxStagedCols) raise(RQ_ERR_UNSUPPORTED, "more than %d columns in one pipeline", kMaxStagedCols);
                            P.col_ptr[P.n_cols] = dc.d; P.col_w[P.n_cols] = (uint8_t)dc.width;
                            staged_of_col[nd.a] = P.n_cols++;
                        }
                        o.kind = S_COL;
                    }
                    o.idx = (uint16_t)staged_of_col[nd.a];
                    leaf_op[i] = o;
                    break;
                }
                case RQ_OP_CONST: { HOpnd o; o.kind = S_IMM; o.imm = nd.imm; leaf_op[i] = o; break; }
                case RQ_OP_CONST_STR: {
                    if (nd.imm < 0 || nd.imm >= plan.strpool_bytes) raise(RQ_ERR_INVALID, "node %d: string offset out of range", i);
                    HOpnd o; o.kind = S_IMM; o.imm = (int64_t)(d_strpool + nd.imm); leaf_op[i] = o; break;
                }
                case RQ_OP_FILTER: use(i, nd.a); break;
                case RQ_OP_SELECT: use(i, nd.a); use(i, nd.b); use(i, nd.c); break;
                case RQ_OP_PROBE: {
                    if (nd.b < 0 || nd.c < 0 || nd.b + nd.c > pl.n_args) raise(RQ_ERR_INVALID, "node %d: probe args out of range", i);
                    for (int k = 0; k < nd.c; k++) { use(i, pl.args[nd.b + k]); sink_ref[pl.args[nd.b + k]] = 1; }
                    break;
                }
                case RQ_OP_PAYLOAD: check_ref(i, nd.a); break;
                case kOpRowId: break;
                case kOpInSet: use(i, nd.a); break;
                default:
                    if (is_binary(nd.op)) { use(i, nd.a); use(i, nd.b); }
                    else raise(RQ_ERR_INVALID, "node %d: unknown op %d", i, nd.op);
            }
        }
        auto sink_use = [&](int ref) {
            if (ref < 0 || ref >= n) raise(RQ_ERR_INVALID, "sink refers to node %d", ref);
            uses[ref]++; last_use[ref] = n; sink_ref[ref] = 1;
        };
        for (int k = 0; k < pl.n_keys; k++) sink_use(pl.keys[k].node);
        for (int k = 0; k < pl.n_vals; k++)
            if (!(pl.sink_kind == RQ_SINK_AGG && pl.vals[k].kind == RQ_AGG_COUNT)) sink_use(pl.vals[k].node);
        // stage layout: one warp tile of every staged column, in source order (tile-major tables:
        // page order), so that adjacent columns of a page arrive with one bulk copy
        {
            std::vector<int> order;       // staged columns
            for (int c = 0; c < P.n_cols; c++) order.push_back(c);
            std::vector<int> src_of(P.n_cols, -1);
            for (size_t k = 0; k < staged_of_col.size(); k++)
                if (src.cols[k].type != RQ_STR && staged_of_col[k] >= 0) src_of[staged_of_col[k]] = (int)k;
            const bool tile_major = src.pax_base != nullptr;
            const bool cross = src.cross[0] != nullptr;    // no runs: the kernel gathers every column itself
            const int n_left = cross ? (int)src.cross[0]->cols.size() : 0;
            P.cross_inner = 0;
            if (tile_major)
                std::sort(order.begin(), order.end(), [&](int a, int b) { return src.cols[src_of[a]].page_off < src.cols[src_of[b]].page_off; });
            uint32_t off = 0;
            P.n_runs = 0;
            for (int c : order) {
                const DevColumn& dc = src.cols[src_of[c]];
                const uint32_t bytes = (uint32_t)kTile * P.col_w[c];
                P.col_off[c] = off;
                const int r = P.n_runs - 1;
                if (cross) {
                    if ((src_of[c] >= n_left) == (src.cross_inner == 1)) P.cross_inner |= 1u << c;
                } else if (tile_major && r >= 0 && P.run_ptr[r] + P.run_bytes[r] == dc.d) {
                    P.run_bytes[r] += bytes;              // adjacent in the page: same copy
                } else {
                    P.run_ptr[P.n_runs] = dc.d;
                    P.run_bytes[P.n_runs] = bytes;
                    P.run_stride[P.n_runs] = (uint32_t)(dc.tile_stride ? dc.tile_stride : (int64_t)bytes);
                    P.run_off[P.n_runs] = off;
                    P.n_runs++;
                }
                off += bytes;
            }
            P.stage_bytes = off;
        }
        derive_bounds();
        // fusion marks
        for (int f = 0; f < n; f++) {
            HOpnd o; int64_t k;
            if (fcmp_of(f, &o, &k)) fused[pl.nodes[f].a] = 1;
        }
        for (int i = 0; i < n; i++) {
            int inner, other; uint8_t gop; int64_t k; HOpnd x;
            if (muli_of(i, &inner, &other, &gop, &k, &x)) fused[inner] = 1;
        }
    }

    // Interval arithmetic over the typed program: column bounds come from the upload statistics,
    // anything that may wrap around int64 becomes "unknown". A value proven to lie in [0, 2^32)
    // has a zero high word, so the 32-bit instruction forms produce identical results.
    void derive_bounds() {
        const __int128 FMIN = INT64_MIN, FMAX = INT64_MAX;
        vlo.assign(n, FMIN); vhi.assign(n, FMAX);
        auto clampset = [&](int i, __int128 lo, __int128 hi) {
            if (lo < FMIN || hi > FMAX) { vlo[i] = FMIN; vhi[i] = FMAX; } else { vlo[i] = lo; vhi[i] = hi; }
        };
        // A tuple reaches the sink only if it passes every selection, so `col CMP const` selections
        // narrow the bounds of the column for everything the sink sees (values computed for tuples that
        // are dropped anyway may fall outside; they are never used).
        std::vector<__int128> clo(n, FMIN), chi(n, FMAX);
        for (int f = 0; f < n; f++) {
            if (pl.nodes[f].op != RQ_OP_FILTER) continue;
            const rq_node& cm = pl.nodes[pl.nodes[f].a];
            int op = cm.op, cn = -1, kn = -1;
            if (op != RQ_OP_LT && op != RQ_OP_LE && op != RQ_OP_GT && op != RQ_OP_GE && op != RQ_OP_EQ) continue;
            if (pl.nodes[cm.a].op == RQ_OP_COL && pl.nodes[cm.b].op == RQ_OP_CONST) { cn = cm.a; kn = cm.b; }
            else if (pl.nodes[cm.a].op == RQ_OP_CONST && pl.nodes[cm.b].op == RQ_OP_COL) {
                cn = cm.b; kn = cm.a;
                op = op == RQ_OP_LT ? RQ_OP_GT : op == RQ_OP_LE ? RQ_OP_GE : op == RQ_OP_GT ? RQ_OP_LT : op == RQ_OP_GE ? RQ_OP_LE : op;
            } else continue;
            const __int128 k = pl.nodes[kn].imm;
            if (op == RQ_OP_LT) chi[cn] = std::min(chi[cn], k - 1);
            else if (op == RQ_OP_LE) chi[cn] = std::min(chi[cn], k);
            else if (op == RQ_OP_GT) clo[cn] = std::max(clo[cn], k + 1);
            else if (op == RQ_OP_GE) clo[cn] = std::max(clo[cn], k);
            else { clo[cn] = std::max(clo[cn], k); chi[cn] = std::min(chi[cn], k); }
        }
        for (int i = 0; i < n; i++) {
            const rq_node& nd = pl.nodes[i];
            switch (nd.op) {
                case RQ_OP_COL: {
                    const DevColumn& dc = src.cols[nd.a];
                    if (dc.type == RQ_STR) break;
                    if (dc.has_stats) { vlo[i] = dc.vmin; vhi[i] = dc.vmax; }
                    else if (dc.type == RQ_I8) { vlo[i] = 0; vhi[i] = 255; }
                    else if (dc.type == RQ_I32) { vlo[i] = INT32_MIN; vhi[i] = INT32_MAX; }
                    if (clo[i] > vlo[i]) vlo[i] = clo[i];
                    if (chi[i] < vhi[i]) vhi[i] = chi[i];
                    if (vlo[i] > vhi[i]) { vlo[i] = vhi[i] = clo[i] > FMIN ? clo[i] : chi[i]; }   // no tuple passes: any bounds do
                    if (vlo[i] < FMIN) vlo[i] = FMIN;
                    if (vhi[i] > FMAX) vhi[i] = FMAX;
                    break;
                }
                case RQ_OP_CONST: vlo[i] = vhi[i] = nd.imm; break;
                case RQ_OP_ADD: clampset(i, vlo[nd.a] + vlo[nd.b], vhi[nd.a] + vhi[nd.b]); break;
                case RQ_OP_SUB: clampset(i, vlo[nd.a] - vhi[nd.b], vhi[nd.a] - vlo[nd.b]); break;
                case RQ_OP_MUL: {
                    const __int128 c[4] = {vlo[nd.a] * vlo[nd.b], vlo[nd.a] * vhi[nd.b], vhi[nd.a] * vlo[nd.b], vhi[nd.a] * vhi[nd.b]};
                    clampset(i, std::min(std::min(c[0], c[1]), std::min(c[2], c[3])), std::max(std::max(c[0], c[1]), std::max(c[2], c[3])));
                    break;
                }
                case RQ_OP_LT: case RQ_OP_LE: case RQ_OP_GT: case RQ_OP_GE: case RQ_OP_EQ: case RQ_OP_NEQ:
                case RQ_OP_EQ_CHAR: case RQ_OP_EQ_VARCHAR: case RQ_OP_NEQ_CHAR: case RQ_OP_NEQ_VARCHAR: case RQ_OP_LIKE:
                    vlo[i] = 0; vhi[i] = 1; break;
                case RQ_OP_AND: case RQ_OP_OR:
                    if (vlo[nd.a] >= 0 && vhi[nd.a] <= 1 && vlo[nd.b] >= 0 && vhi[nd.b] <= 1) { vlo[i] = 0; vhi[i] = 1; }
                    break;
                case RQ_OP_SELECT:
                    vlo[i] = std::min(vlo[nd.b], vlo[nd.c]); vhi[i] = std::max(vhi[nd.b], vhi[nd.c]); break;
                case kOpInSet: vlo[i] = 0; vhi[i] = 1; break;
                default: break;   // DIV, PROBE, PAYLOAD, strings: unknown
            }
        }
    }
    bool is_u32(int node) const { return vlo[node] >= 0 && vhi[node] <= 0xffffffffLL; }

    bool is_col8(int node) const {
        return pl.nodes[node].op == RQ_OP_COL && leaf_op[node].kind == S_COL && P.col_w[leaf_op[node].idx] == 8;
    }

    // FILTER(COL cmp CONST) where the compare has no other consumer: one unit that only narrows
    // the selection mask. 4- and 1-byte columns compare in 32 bits, so the constant must fit (it
    // always does for dates / flags; otherwise the generic form is used). Returns the D_LT..D_NE
    // compare with the column on the left.
    int fcmp_of(int f, HOpnd* col, int64_t* imm) const {
        const rq_node& fl = pl.nodes[f];
        if (fl.op != RQ_OP_FILTER) return 0;
        const rq_node& cm = pl.nodes[fl.a];
        if (uses[fl.a] != 1 || sink_ref[fl.a]) return 0;
        if (!fcmp_left(cm.op)) return 0;
        const int xo = pl.nodes[cm.a].op, yo = pl.nodes[cm.b].op;
        int code = 0, cn = -1, kn = -1;
        if (xo == RQ_OP_COL && yo == RQ_OP_CONST) { code = fcmp_left(cm.op); cn = cm.a; kn = cm.b; }
        else if (xo == RQ_OP_CONST && yo == RQ_OP_COL) { code = fcmp_right(cm.op); cn = cm.b; kn = cm.a; }
        else return 0;
        const HOpnd o = leaf_op[cn];
        if (o.kind != S_COL) return 0;
        const int64_t k = leaf_op[kn].imm;
        if (P.col_w[o.idx] != 8 && (k < INT32_MIN || k > INT32_MAX)) return 0;
        *col = o; *imm = k;
        return code;
    }

    // MUL(ADD/SUB(col8, const), other) where the inner node has no other consumer:
    // t = (x GOP imm) * other in one unit (TPC-H's  price * (1 - discount) * (1 + tax)  shapes)
    bool muli_of(int i, int* inner, int* other, uint8_t* gop, int64_t* k, HOpnd* x) const {
        const rq_node& nd = pl.nodes[i];
        if (nd.op != RQ_OP_MUL || nd.a == nd.b) return false;
        for (int side = 0; side < 2; side++) {
            const int j = side == 0 ? nd.a : nd.b, o = side == 0 ? nd.b : nd.a;
            const rq_node& in = pl.nodes[j];
            if ((in.op != RQ_OP_ADD && in.op != RQ_OP_SUB) || uses[j] != 1 || sink_ref[j]) continue;
            if (is_leaf(pl.nodes[o].op) && !is_col8(o)) continue;     // other side: 64-bit column or a slot
            uint8_t g = 0; int cn = -1, kn = -1;
            if (is_col8(in.a) && pl.nodes[in.b].op == RQ_OP_CONST) { cn = in.a; kn = in.b; g = in.op == RQ_OP_ADD ? D_ADD : D_SUB; }
            else if (pl.nodes[in.a].op == RQ_OP_CONST && is_col8(in.b)) { cn = in.b; kn = in.a; g = in.op == RQ_OP_ADD ? D_ADD : D_RSUB; }
            else continue;
            *inner = j; *other = o; *gop = g; *k = leaf_op[kn].imm; *x = leaf_op[cn];
            return true;
        }
        return false;
    }
};

}  // namespace

#include "engine_exec.inl"
#include "tbl_loader.inl"
