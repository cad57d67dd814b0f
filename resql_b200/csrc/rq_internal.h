// Internal (host+device) definitions of the resql_b200 engine. Not part of the ABI.
#pragma once
#include <stdint.h>
#include <stddef.h>

namespace rq {

// ---- geometry of the scan kernel ------------------------------------------------------------
// Every WARP is an independent pipeline: it owns a ring of TMA stages in shared memory, each
// holding one warp tile (256 tuples of every scanned column), and interprets the program over
// a register tile of 8 tuples per lane. Lane l owns tuples {64k + 2l, 64k + 2l + 1 : k=0..3} of
// the tile, so every operand fetch is a conflict-free 16/8/2-byte vector load.
constexpr int kR          = 8;                  // tuples per lane per tile
constexpr int kTile       = 32 * kR;            // 256 tuples per warp tile
constexpr int kPadRows    = 1024;               // owned tables are padded to this many rows
constexpr int kMaxStages  = 4;                  // TMA ring depth per warp
constexpr int kMaxWarps   = 16;                 // warps per CTA (one persistent CTA per SM)

constexpr int kMaxStagedCols = 16;
constexpr int kMaxStrCols    = 8;
constexpr int kMaxInsn       = 128;
constexpr int kMaxKeys       = 8;
constexpr int kMaxAggs       = 16;
constexpr int kMaxOut        = 24;
constexpr int kMaxLateOut    = 64;     // output columns of a late-materialized pipeline (IMPL_LATE) and of a result
constexpr int kMaxImm        = 32;
constexpr int kMaxProbes     = 4;
constexpr int kMaxSlots      = 12;
constexpr int kNAR           = 6;      // aggregates held in registers per group (register path)
constexpr int kRegGroups     = 4;      // groups held in registers per warp (register path)
constexpr int kLowCardMaxGroups = 8;   // groups per warp with lane-private shared-memory accumulators
constexpr int kGroupTableCap = 2048;   // global table of the low-cardinality aggregate paths

// register-path accumulation forms of a SUM aggregate (chosen on the host from the value bounds)
enum AggMode : uint8_t { AM_FULL = 0, AM_P1 = 1, AM_P2 = 2, AM_W64 = 3 };
// what the aggregate loop of the register path does for one aggregate (KParams::agg_desc bits 0-2)
enum AggForm : uint32_t { AF_NONE = 0, AF_P1 = 1, AF_P2 = 2, AF_W64 = 3, AF_FULL = 4, AF_MIN = 5, AF_MAX = 6 };

enum SinkImpl { IMPL_LOWAGG = 1, IMPL_HASHAGG = 2, IMPL_BUILD = 3, IMPL_EMIT = 4, IMPL_REGAGG = 5, IMPL_GROUPJOIN = 6,
                IMPL_LATE = 7 };   // IMPL_EMIT of a record of references, then rq_late_gather (engine_exec.inl)

// ---- status words of a pipeline launch ----------------------------------------------------------
// One block in device memory (Engine::flags, 64 bytes) that kernels raise and count into, and its
// pinned host copy the host reads back after a launch.
struct FlagBlock {
    int32_t  overflow;      // a warp met more groups than its aggregation path tracks
    int32_t  ht_full;       // hash table full, or past the load a launch may add
    int32_t  err;           // 1: division by zero, 2: probe in a kernel variant without probe code
    int32_t  dup_key;       // direct-address build: duplicate key, or a key outside the domain
    uint64_t dup_matches;   // multi-match probe: tuples with more than one match
    uint64_t entries;       // hash / direct-address table entries the launch added
    uint64_t extra;         // a device word copied behind the flags so one read brings both
    uint64_t reserved;
    uint64_t popcount;      // shared build: set bits of the all-reduced bitmap
};
#ifndef __CUDACC_RTC__     // (NVRTC has no offsetof: a run-time compiled kernel, jit.h, gets the one word index it uses below)
static_assert(offsetof(FlagBlock, overflow) == 0, "FlagBlock layout");
static_assert(offsetof(FlagBlock, ht_full) == 4, "FlagBlock layout");
static_assert(offsetof(FlagBlock, err) == 8, "FlagBlock layout");
static_assert(offsetof(FlagBlock, dup_key) == 12, "FlagBlock layout");
static_assert(offsetof(FlagBlock, dup_matches) == 16, "FlagBlock layout");
static_assert(offsetof(FlagBlock, entries) == 24, "FlagBlock layout");
static_assert(offsetof(FlagBlock, extra) == 32, "FlagBlock layout");
static_assert(offsetof(FlagBlock, reserved) == 40, "FlagBlock layout");
static_assert(offsetof(FlagBlock, popcount) == 48, "FlagBlock layout");
static_assert(sizeof(FlagBlock) <= 64, "FlagBlock must fit Engine::flags");
// The words in front of `extra` are cleared before a launch and, for a shared build, summed over
// the ranks as four uint64.
constexpr size_t kFlagsCleared = offsetof(FlagBlock, extra);
static_assert(kFlagsCleared == 32, "the cleared and summed prefix is four uint64");
// int32 word indices, for device code that addresses the block through an int32_t*
constexpr int kFlagWordErr      = offsetof(FlagBlock, err) / 4;
constexpr int kFlagWordDupKey   = offsetof(FlagBlock, dup_key) / 4;
constexpr int kFlagWordEntries  = offsetof(FlagBlock, entries) / 4;
constexpr int kFlagWordPopcount = offsetof(FlagBlock, popcount) / 4;
// KParams::ht_full points at FlagBlock::ht_full; the direct-address build raises dup_key through it
constexpr int kDupKeyFromHtFull = (offsetof(FlagBlock, dup_key) - offsetof(FlagBlock, ht_full)) / 4;
static_assert(kDupKeyFromHtFull == 2, "the NVRTC value below");
#else
constexpr int kDupKeyFromHtFull = 2;
#endif

// ---- operation codes shared by the host-level program and the device encoding ----------------
enum DOp : uint8_t {
    D_LD = 1, D_ADD, D_SUB, D_RSUB, D_MUL, D_DIV, D_RDIV, D_AND, D_OR,
    D_LT, D_LE, D_GT, D_GE, D_EQ, D_NE,
    D_EQC, D_EQV, D_NEC, D_NEV, D_LIKE, D_RLIKE,
    D_SEL,
    D_INSET         // U_GEN: t = (x in the constant set at imm), see InSetHeader
};

enum DSrc : uint8_t { S_NONE = 0, S_COL = 1, S_SLOT = 2, S_IMM = 3, S_STR = 4 };

// ---- device-level instruction -------------------------------------------------------------------
// The program is a memory-to-memory vector VM over the warp's shared-memory region: every unit
// reads its operands from staged columns / value slots (or an immediate), computes 8 tuples per
// lane in registers and writes the result to a slot and/or folds it into the selection mask.
// Nothing but the selection mask lives in registers across units, so the one big switch costs no
// register shuffling. Opcode and operand form are fused into `code` on the host and operands are
// precomputed byte offsets, so a unit does no address bookkeeping per tuple.
enum UKind : uint8_t {             // operand kinds
    K_NONE = 0, K_M64, K_M32, K_M8, K_IMM, K_STR,
    K_IMM2        // constant in KParams::imm[offset] (second constant of a unit)
};

#define RQ_BINOPS(X) X(ADD) X(SUB) X(RSUB) X(MUL) X(AND) X(OR) X(LT) X(LE) X(GT) X(GE) X(EQ) X(NE)

enum UCode : uint8_t {
    U_END = 0,
    // t = x OP y (64-bit operands in shared memory) | t = x OP imm
#define RQ_X(N) U_##N##_MM, U_##N##_MI,
    RQ_BINOPS(RQ_X)
#undef RQ_X
    U_MULADDI, U_MULSUBI, U_MULRSUBI,   // t = (x + imm) * y | (x - imm) * y | (imm - x) * y
    // the same, and x * y, when both factors are proven to lie in [0, 2^32): one IMAD.WIDE.U32
    U_MULADDI32, U_MULSUBI32, U_MULRSUBI32, U_MUL32_MM,
    U_GEN,                              // t = gop(x, y [, z]) with operands of any kind
    // valid &= (column CMP imm): selection-fused compares, nothing stored
    U_FLT_M64, U_FLE_M64, U_FGT_M64, U_FGE_M64, U_FEQ_M64, U_FNE_M64,
    U_FLT_M32, U_FLE_M32, U_FGT_M32, U_FGE_M32, U_FEQ_M32, U_FNE_M32,
    U_FLT_M8,  U_FLE_M8,  U_FGT_M8,  U_FGE_M8,  U_FEQ_M8,  U_FNE_M8,
    // valid &= (imm <= column <= imm + span): two selection compares on one column fused
    U_FRANGE_M64, U_FRANGE_M32, U_FRANGE_M8,
    U_PROBE
};

constexpr uint8_t UF_XSLOT  = 1;   // x offset is relative to the warp region (a slot), else the stage
constexpr uint8_t UF_YSLOT  = 2;
constexpr uint8_t UF_ZSLOT  = 4;
constexpr uint8_t UF_FILTER = 8;   // valid &= (t & 0xff) != 0   (selection.h:62-66)
constexpr uint8_t UF_STORE  = 16;  // t goes to the slot at dstrel

// Fully decoded on the host; the CTA copies the program to shared memory once and every unit is
// fetched with two broadcast 128-bit loads.
struct UInsn {
    uint8_t  code;
    uint8_t  flags;
    uint8_t  gop;       // U_GEN: DOp
    uint8_t  aux;       // probe index
    uint8_t  xkind, ykind, zkind, pad;   // U_GEN: UKind of the operands
    uint32_t xrel;      // byte offset of x (stage- or region-relative); K_STR: string column
    uint32_t dstrel;    // byte offset of the destination slot inside the warp region
    int64_t  imm;       // immediate operand / compare constant / range low bound
    uint32_t yrel;      // byte offset of y                 } selection-fused range compare:
    uint32_t zrel;      // byte offset of z; K_IMM: index   } yrel|zrel<<32 = span (unsigned)
};
static_assert(sizeof(UInsn) == 32, "UInsn must be 32 bytes");

// ---- constant sets of IN lists (U_GEN D_INSET) -----------------------------------------------------
// A set is one block of 64-bit words in device memory, built on the host (engine_exec.inl "IN lists"):
// the header, then the data of its form.
//   IS_BITMAP   integers: bit (x - a) of 32-bit words over [a, a + b]        one range test, one load
//   IS_SORTED   integers: a sorted values                                    branchless binary search
//   IS_CHAR     strings: open-addressing table of cap = a + 1 entries {hash, byte offset of the
//   IS_VARCHAR  constant from the block start (0 = empty)}, then the NUL-terminated constants
enum InSetForm : uint32_t { IS_BITMAP = 0, IS_SORTED = 1, IS_CHAR = 2, IS_VARCHAR = 3 };
struct InSetHeader {
    uint64_t form;
    uint64_t a;          // IS_BITMAP: lowest value; IS_SORTED: count; IS_CHAR / IS_VARCHAR: table mask
    uint64_t b;          // IS_BITMAP: highest value - lowest value
    uint64_t pad;
};
static_assert(sizeof(InSetHeader) == 32, "the set data starts at word 4");

// Hash of a string constant of a set and of a tuple's string: FNV-1a over the bytes in front of the
// NUL; CHAR sets (`blank_pad`) leave out trailing blanks, which compareChar ignores.
#ifdef __CUDACC__
__host__ __device__
#endif
inline uint64_t inset_str_hash(const char* s, bool blank_pad) {
    int n = 0;
    while (s[n] != '\0') n++;
    if (blank_pad) while (n > 0 && s[n - 1] == ' ') n--;
    uint64_t h = 0xcbf29ce484222325ULL;
    for (int i = 0; i < n; i++) { h ^= (unsigned char)s[i]; h *= 0x100000001b3ULL; }
    return h;
}

struct VRef {           // value reference used by sinks (keys, payloads, outputs)
    uint8_t  kind;      // UKind
    uint8_t  slot;      // bit0: offset relative to the warp region; bit1: value fits in unsigned 32 bits
    uint16_t off16;     // byte offset >> 4; K_IMM: index into KParams::imm; K_STR: string column
};

// hash table used by joins (build then probe in separate kernels) and by hash aggregation
struct DHashTable {
    uint64_t  cap_mask;     // capacity - 1 (power of two)
    uint32_t  shift;        // home slot = hash >> shift  (64 - log2(capacity): the high hash bits)
    uint32_t  bloom_mask;   // words - 1 of the blocked Bloom filter (joins), 0 = none
    // hash of a single integer key: (key - hsub) * hmul. Fibonacci hashing (hsub 0, hmul golden ratio)
    // by default; for a dense key domain [lo, hi] known from the upload statistics the ORDER-PRESERVING
    // form hsub = lo, hmul = floor((2^64 - 1) / (hi - lo + 1)): neighbouring keys land in neighbouring
    // slots, so a build or probe that visits keys in (nearly) sorted order - orders by
    // o_orderkey, lineitem by l_orderkey - streams through the table instead of hopping over HBM.
    uint64_t  hmul;
    int64_t   hsub;
    uint32_t  bloom_shift;  // reserved (0): Bloom word index always comes from the mixed hash
    uint32_t  pad2_;
    uint64_t  limit;        // entries a launch may add before it raises the table-full flag
    uint32_t* bloom;        // 32-bit blocks, two bits per key; sized to stay L2 resident
    // entries are packed rows: [tag][nk key words][nv payload / accumulator words], padded to a
    // multiple of 4 words, so that a hit costs one memory round trip (tag 0 = empty, 1 = being
    // written, else hash | 2)
    uint64_t* ent;
    uint32_t  stride;       // words per entry
    uint32_t  pad_;
    int32_t   nk, nv;
    uint8_t   key_kind[kMaxKeys];   // 0 integer, 1 CHAR, 2 VARCHAR
    // DIRECT-ADDRESS form (join builds on one integer key whose value domain [dlo, dlo + dsize) is
    // known and dense enough, keys unique): no slots, no tags, no walks. A bitmap says which keys are
    // present (exact semi-join filter, a few MB: L2 resident), payload word q of key k lives at
    // darr[(k - dlo) * dnv + q]. A build is a plain store per tuple, a probe one bit test and at
    // most one payload fetch. Duplicate keys raise a flag and the host rebuilds the hash form.
    uint32_t  packed;               // hash aggregation: entry = [packed group key + 1][accumulators] (no tag, no key words)
    uint32_t  pad3_;
    uint32_t  direct;
    uint32_t  dnv;                  // words per key: payloads, then groupjoin accumulators (KParams::gj_acc_word)
    int64_t   dlo;
    uint64_t  dsize;
    uint32_t* dbits;
    uint64_t* darr;
};

struct DProbe {
    DHashTable ht;
    VRef       key[kMaxKeys];
    uint8_t    out_slot[kMaxOut];   // payload column k -> slot (0xff = not needed)
    uint8_t    pay_word[kMaxOut];   // payload column k -> word of the entry that holds it (a key word when the
                                    // payload repeats a join key)
    int32_t    n_out;
    int32_t    single;
    int32_t    bloom_only;          // semi-join reduction only: no table walk, no payload
    int32_t    fetch;               // key[0] is the entry index of a match found by an expansion pass
    unsigned long long* dup_counter;   // counts tuples with more than one match (multi-match mode)
};

struct KParams {
    // source
    int64_t        n_rows;
    const int64_t* n_rows_ptr;          // if non-null the row count is read on the device
    int64_t        n_rows_cap;          // ... and clamped to the rows the source has room for
    int32_t        borrowed;            // source buffers may end exactly at n_rows (no padding)
    int32_t        stream_hint;         // mark scanned data evict-first in L2
    int32_t        l2_prefetch;         // pull the next tile into L2 while the current one is processed
                                        // (pure scans only: pipelines with hash structures want L2 for those)
    int32_t        pad0_;
    const uint32_t* tile_range;         // if non-null: only tiles [tile_range[0], tile_range[1]) are scanned
    int32_t        n_cols;              // staged (TMA) columns
    // A tile is staged by one bulk copy per RUN: a contiguous byte range of the source that holds
    // the tile's chunk of one column (plain column arrays) or of several adjacent columns (tables
    // owned by the engine are stored tile-major, see engine.cu "storage layout").
    int32_t        n_runs;
    const unsigned char* run_ptr[kMaxStagedCols];   // the run of tile 0
    uint32_t       run_bytes[kMaxStagedCols];       // bytes per tile
    uint32_t       run_stride[kMaxStagedCols];      // distance between the runs of consecutive tiles
    uint32_t       run_off[kMaxStagedCols];         // destination offset inside a stage
    const unsigned char* col_ptr[kMaxStagedCols];   // plain column arrays only (guarded tail of borrowed sources)
    uint32_t       col_off[kMaxStagedCols];   // byte offset inside a stage
    uint8_t        col_w[kMaxStagedCols];     // 1, 4, 8
    int32_t        n_strcols;
    const unsigned char* str_ptr[kMaxStrCols];
    uint32_t       str_w[kMaxStrCols];
    uint32_t       stage_bytes;         // kTile * sum(col_w)
    int32_t        stages;              // TMA ring depth per warp
    // shared memory carve-up: [mbarriers][warp 0 region][warp 1 region]...
    uint32_t       warp_off;            // byte offset of warp 0's region
    uint32_t       warp_bytes;          // bytes per warp region
    uint32_t       slots_rel;           // slots, relative to the warp region
    uint32_t       acc_rel;             // lane-private accumulators (shared-memory path)
    uint32_t       prog_off;            // byte offset of the program copy
    uint32_t       smem_bytes;          // total dynamic shared memory of the CTA
    int32_t        n_slots;
    int32_t        warps;               // warps per CTA
    // program
    int32_t        n_insn;
    UInsn          insn[kMaxInsn];
    int64_t        imm[kMaxImm];
    // grouping / aggregation
    int32_t        nk;
    VRef           key[kMaxKeys];
    uint8_t        key_shift[kMaxKeys]; // packed group key: sum((value & mask) << shift)
    uint8_t        key_bits[kMaxKeys];
    int32_t        key32;               // the packed key fits in 32 bits
    int32_t        na;
    uint8_t        agg_kind[kMaxAggs];
    VRef           agg_src[kMaxAggs];    // aggregate inputs (COUNT has none)
    uint8_t        agg_mode[kMaxAggs];   // register path: AggMode of a SUM
    uint8_t        agg_shift[kMaxAggs];  // AM_P2: bits of the low piece
    int32_t        flush_tiles;          // register path: flush the 32-bit piece sums every this many tiles (0 = never)
    int32_t        pad1_;
    uint32_t       agg_desc[kMaxAggs];   // register path: AggForm | operand location, see the aggregate loop
    int32_t        G;                    // lane-private groups per warp (shared-memory path)
    // low-card global table (packed key)
    uint32_t*      g_state;              // [kGroupTableCap]
    int64_t*       g_keys;               // [kGroupTableCap]
    int64_t*       g_acc;                // [kGroupTableCap][kMaxAggs]
    int32_t*       overflow;             // set when a warp meets more groups than its path tracks
    // hash aggregate / build
    DHashTable     ht;
    int32_t*       ht_full;              // set when the table is full
    unsigned long long* ht_entries;      // entries added by this launch
    // groupjoin (IMPL_GROUPJOIN): ht is the probed direct-address table; the aggregates of a tuple go
    // into words [gj_acc_word, + na) of the entry its key selects. A direct-address build writes the
    // identities of agg_kind[0 .. na) into those words of every entry it stores.
    uint32_t*      gj_touched;           // bit per entry: it received a tuple
    uint32_t       gj_acc_word;
    int32_t        pad2_;
    // probes
    int32_t        n_probes;
    DProbe         probe[kMaxProbes];
    // materialize
    int32_t        sink;                 // SinkImpl executed after the units of every tile
    int32_t        expand_probe;         // IMPL_EMIT: >= 0 = emit one row per match of this probe, with the
                                         // entry index of the match as an extra last column
    int32_t        n_out;
    VRef           out[kMaxOut];
    int64_t*       out_col[kMaxOut];
    unsigned long long* out_count;
    int64_t        out_cap;
    // runtime error flag (division by zero)
    int32_t*       err;
    // nested-loops join source (RQ_SRC_CROSS, kernel variant CROSS): pair p of the source is (row
    // p / n_inner of the outer relation, row p % n_inner of the inner one); every staged column is a
    // plain int64 array col_ptr[c] of one of the two. (Behind every other field, so that the variants
    // without it address their parameters exactly as before.)
    const int64_t* cross_rows[2];        // [outer, inner]: row counts, read on the device ...
    int64_t        cross_cap[2];         // ... and clamped to the rows each relation has room for
    uint32_t       cross_inner;          // bit c: staged column c belongs to the inner relation
    int32_t        pad3_;
    // late materialization (kernel variant LATE, engine_exec.inl "late materialization"): before the
    // program of a tile runs, the absolute row (pair) index of every tuple is written to the slot at
    // late_row_rel (late_row != 0); probe p writes the reference of its matched entry (hash slot index,
    // or key - dlo of a direct-address table) to slot late_ref_slot[p] (0xff: none). (Behind every other
    // field, like the cross fields.)
    int32_t        late_row;
    uint32_t       late_row_rel;
    uint8_t        late_ref_slot[kMaxProbes];
    int32_t        late;                 // launch the LATE variant
    // sink rounds (kernel variant ROUNDS, materialize only; engine_exec.inl "sink rounds"): units
    // [0, prefix_end) are the prefix, which holds every filter and probe; after it the tile's output
    // positions are located once. Round k then runs units [round_unit_end[k - 1], round_unit_end[k])
    // (the first round starts at prefix_end) and stores values [round_val_end[k - 1], round_val_end[k])
    // into their output columns. (Behind every other field, like the cross and late fields.)
    int32_t        n_rounds;             // 0: the pipeline has the single sink of the other variants
    int32_t        prefix_end;
    uint16_t       round_unit_end[kMaxLateOut];
    uint8_t        round_val_end[kMaxLateOut];
    VRef           rval[kMaxLateOut];    // the sink values, in value (= output column) order
    int64_t*       rout_col[kMaxLateOut];
};

}  // namespace rq
