// Fused scan -> filter -> project -> (probe | aggregate | build | materialize) kernel for sm_100a.
//
// One persistent CTA per SM; every WARP is an independent pipeline. A warp owns a ring of TMA
// stages in shared memory (cp.async.bulk + one mbarrier per stage); each stage holds one warp
// tile = 256 tuples of every scanned column. Per tile the warp
//   1. runs the typed program: a memory-to-memory vector VM over its shared-memory region. Every
//      unit reads operands from staged columns / value slots, computes 8 tuples per lane and
//      writes a slot and/or narrows the selection mask. ONE switch per unit (opcode and operand
//      form fused on the host, operands are precomputed offsets); only the selection mask lives in
//      registers across units, so the switch causes no register shuffling;
//   2. runs the sink as straight-line code: group match + aggregation, hash aggregation,
//      hash-join build, or materialize;
//   3. re-arms the stage. No CTA-wide barrier exists in the steady state.
// Staging is done by named pieces: issue_tile (the bulk copies of one stage), stage_tile (wait, or
// stage the guarded tail of a borrowed source, or the pairs of a cross source), prefetch_next (L2
// prefetch of the next tile) and drain_ring (early exit on a full hash table). Repeated sink pieces
// have one definition each: atomic_agg (hash aggregation and groupjoin), put_match (probe matches),
// warp_group_slot (group-table slot of a flush), flush_groups (the groups a flush covers), leader_key
// (a new dictionary key), reg_at / reg_set (an element of a register array). The materialize sink
// (sink_emit, made of emit_locate and the stores) and the LOWAGG end flush (flush_lowagg) are functions;
// the program, the probe unit and the other sinks are written in the kernel body (DESIGN §3.1). The
// round variant (ROUNDS) runs the program in pieces around emit_locate and emit_put.
//
// Aggregation (template parameter GR):
//   GR = 1 / 4  register path: up to GR groups x kNAR aggregates live in registers for the whole
//               kernel; a tuple is added to every group accumulator through a 0/1 multiplier
//               (IMAD.WIDE.U32 on the FMA pipe, no shared-memory traffic, no dependent chain).
//   GR = 0      generic sinks: lane-private shared-memory accumulators for up to 8 groups per
//               warp, HBM hash aggregation, hash-join build, materialize.
//
// Semantics restated from the reference (Henning1/resql):
//   arithmetic / compares  src/ExpressionsJitFlounder.h:298-689
//   selection              src/operators/selection.h:52-70
//   aggregation            src/operators/aggregation.h:95-152, :240-295
//   hash join              src/operators/hashjoin.h:118-279
//   string compares        src/qlib/scalar.h:16-120
#pragma once
#include <cuda_runtime.h>
#include "../../include/resql_b200.h"
#include "rq_internal.h"
#include "device_util.cuh"
#include "hash_kernels.cuh"

namespace rq {

constexpr unsigned kFull = 0xffffffffu;

// tuple r of lane l sits at row 64*(r/2) + 2*l + (r%2) of the warp tile
__device__ __forceinline__ int row_in_tile(int r, int lane) {
    return (r >> 1) * 64 + 2 * lane + (r & 1);
}

// ---- shared memory through 32-bit shared-space addresses --------------------------------------
// (explicit ld.shared / st.shared: no generic-address arithmetic per access; volatile keeps the
// program order between a slot store and the loads of later units)
__device__ __forceinline__ void lds_v2b64(uint32_t a, int64_t& x, int64_t& y) {
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(x), "=l"(y) : "r"(a));
}
__device__ __forceinline__ void sts_v2b64(uint32_t a, int64_t x, int64_t y) {
    asm volatile("st.shared.v2.b64 [%0], {%1, %2};" ::"r"(a), "l"(x), "l"(y) : "memory");
}
__device__ __forceinline__ void lds_v2b32(uint32_t a, int32_t& x, int32_t& y) {
    asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(x), "=r"(y) : "r"(a));
}
__device__ __forceinline__ void lds_v2u8(uint32_t a, uint32_t& x, uint32_t& y) {
    asm volatile("ld.shared.v2.u8 {%0, %1}, [%2];" : "=r"(x), "=r"(y) : "r"(a));
}
__device__ __forceinline__ uint4 lds_v4b32(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_b32(uint32_t a, uint32_t v) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ int64_t lds_b64(uint32_t a) {
    int64_t v; asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v) : "r"(a)); return v;
}
__device__ __forceinline__ int32_t lds_s32(uint32_t a) {
    int32_t v; asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a)); return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) {
    uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v;
}
__device__ __forceinline__ void sts_b64(uint32_t a, int64_t v) {
    asm volatile("st.shared.b64 [%0], %1;" ::"r"(a), "l"(v) : "memory");
}
__device__ __forceinline__ void sts_u8(uint32_t a, uint32_t v) {
    asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

// register tile <-> shared memory; `a` already includes the lane offset (16 / 8 / 2 bytes per lane)
__device__ __forceinline__ void ld_m64(uint32_t a, int64_t (&v)[kR]) {
#pragma unroll
    for (int k = 0; k < kR / 2; k++) lds_v2b64(a + k * 512, v[2 * k], v[2 * k + 1]);
}
__device__ __forceinline__ void st_m64(uint32_t a, const int64_t (&v)[kR]) {
#pragma unroll
    for (int k = 0; k < kR / 2; k++) sts_v2b64(a + k * 512, v[2 * k], v[2 * k + 1]);
}
__device__ __forceinline__ void ld_m32(uint32_t a, int32_t (&v)[kR]) {
#pragma unroll
    for (int k = 0; k < kR / 2; k++) lds_v2b32(a + k * 256, v[2 * k], v[2 * k + 1]);
}
__device__ __forceinline__ void ld_m8(uint32_t a, uint32_t (&v)[kR]) {
#pragma unroll
    for (int k = 0; k < kR / 2; k++) lds_v2u8(a + k * 64, v[2 * k], v[2 * k + 1]);
}

struct WarpCtx {
    uint32_t stage;     // shared address of the current stage (columns of the current tile)
    uint32_t wbase;     // shared address of this warp's region
    int64_t  row0;      // first tuple of the tile in the source
    int      lane;
};

// ---- what the host knows at launch ------------------------------------------------------------
// The kernel reads every field that stays the same across executions of a pipeline on the same
// tables (program encoding, operand kinds and offsets, sink descriptors, stage layout, probe flags)
// through a spec type. GenericSpec reads them from KParams at run time; that is what the
// ahead-of-time kernels use. A specialization compiled at run time (jit.h) provides the same
// accessors as constants, so the unit switch, the operand-kind dispatch and the sink's form branches
// fold away. Pointers, row counts, tile ranges, capacities and immediates are always read from KParams.
// The baked fields: F(type, accessor, value) for a scalar, A(type, accessor, length, value of element i)
// for an array, PR / PR2 the same per probe p (jit.h generates a specialization from this list).
#define RQ_SPEC_FIELDS(F, A, PR, PR2)                                                                         \
    F(int, n_insn, P.n_insn) F(int, sink, P.sink) F(int, na, P.na) F(int, nk, P.nk) F(int, key32, P.key32)    \
    F(int, G, P.G) F(int, expand_probe, P.expand_probe) F(int, n_out, P.n_out)                               \
    F(int, n_cols, P.n_cols) F(int, n_runs, P.n_runs) F(int, stages, P.stages)                               \
    F(uint32_t, stage_bytes, P.stage_bytes) F(uint32_t, warp_off, P.warp_off) F(uint32_t, warp_bytes, P.warp_bytes) \
    F(uint32_t, slots_rel, P.slots_rel) F(uint32_t, acc_rel, P.acc_rel) F(uint32_t, prog_off, P.prog_off)     \
    F(int, l2_prefetch, P.l2_prefetch) F(int, stream_hint, P.stream_hint)                                    \
    F(uint32_t, ht_direct, P.ht.direct) F(uint32_t, ht_packed, P.ht.packed) F(int, ht_nk, P.ht.nk)            \
    A(int, ht_key_kind, kMaxKeys, P.ht.key_kind[i])                                                          \
    A(VRef, key, kMaxKeys, P.key[i]) A(int, key_shift, kMaxKeys, P.key_shift[i]) A(int, key_bits, kMaxKeys, P.key_bits[i]) \
    A(int, agg_kind, kMaxAggs, P.agg_kind[i]) A(int, agg_mode, kMaxAggs, P.agg_mode[i])                      \
    A(int, agg_shift, kMaxAggs, P.agg_shift[i]) A(uint32_t, agg_desc, kMaxAggs, P.agg_desc[i])                \
    A(VRef, agg_src, kMaxAggs, P.agg_src[i]) A(VRef, out, kMaxOut, P.out[i])                                  \
    A(uint32_t, run_off, kMaxStagedCols, P.run_off[i]) A(uint32_t, run_bytes, kMaxStagedCols, P.run_bytes[i])  \
    A(uint32_t, run_stride, kMaxStagedCols, P.run_stride[i])                                                 \
    A(uint32_t, col_off, kMaxStagedCols, P.col_off[i]) A(int, col_w, kMaxStagedCols, P.col_w[i])              \
    PR(int, pr_fetch, pr.fetch) PR(uint32_t, pr_direct, pr.ht.direct)                         \
    PR(int, pr_bloom_only, pr.bloom_only) PR(int, pr_single, pr.single)                       \
    PR(int, pr_n_out, pr.n_out) PR(int, pr_nk, pr.ht.nk) PR(bool, pr_bloom, pr.ht.bloom != nullptr) \
    PR2(int, pr_key_kind, kMaxKeys, pr.ht.key_kind[i]) PR2(VRef, pr_key, kMaxKeys, pr.key[i]) \
    PR2(int, pr_out_slot, kMaxOut, pr.out_slot[i]) PR2(int, pr_pay_word, kMaxOut, pr.pay_word[i])
struct GenericSpec {
    static constexpr bool kFixed = false;
    // unit pc of the program, from its copy in shared memory at `prog`
    static __device__ __forceinline__ UInsn insn(const KParams&, uint32_t prog, int pc) {
        const uint4 w0 = lds_v4b32(prog + pc * 32), w1 = lds_v4b32(prog + pc * 32 + 16);
        UInsn in;
        in.code = (uint8_t)w0.x; in.flags = (uint8_t)(w0.x >> 8); in.gop = (uint8_t)(w0.x >> 16); in.aux = (uint8_t)(w0.x >> 24);
        in.xkind = (uint8_t)w0.y; in.ykind = (uint8_t)(w0.y >> 8); in.zkind = (uint8_t)(w0.y >> 16);
        in.xrel = w0.z; in.dstrel = w0.w;
        in.imm = (int64_t)((uint64_t)w1.x | ((uint64_t)w1.y << 32));
        in.yrel = w1.z; in.zrel = w1.w;
        return in;
    }
#define RQ_SPEC_FIELD(T, NAME, EXPR) static __device__ __forceinline__ T NAME(const KParams& P) { return EXPR; }
#define RQ_SPEC_ARRAY(T, NAME, N, EXPR) static __device__ __forceinline__ T NAME(const KParams& P, int i) { return EXPR; }
#define RQ_SPEC_PROBE(T, NAME, EXPR) static __device__ __forceinline__ T NAME(const DProbe& pr, int) { return EXPR; }
#define RQ_SPEC_PROBE2(T, NAME, N, EXPR) static __device__ __forceinline__ T NAME(const DProbe& pr, int, int i) { return EXPR; }
    RQ_SPEC_FIELDS(RQ_SPEC_FIELD, RQ_SPEC_ARRAY, RQ_SPEC_PROBE, RQ_SPEC_PROBE2)
#undef RQ_SPEC_FIELD
#undef RQ_SPEC_ARRAY
#undef RQ_SPEC_PROBE
#undef RQ_SPEC_PROBE2
};

// any operand kind -> 8 int64 values (rare forms, group keys, aggregate inputs)
__device__ __forceinline__ void fetch(const KParams& P, const WarpCtx& c, int kind, bool slot,
                                      uint32_t off, int64_t imm, int64_t (&v)[kR]) {
    const uint32_t base = (slot ? c.wbase : c.stage) + off;
    switch (kind) {
        case K_M64: ld_m64(base + c.lane * 16, v); break;
        case K_M32: {
            int32_t t[kR]; ld_m32(base + c.lane * 8, t);
#pragma unroll
            for (int r = 0; r < kR; r++) v[r] = t[r];
            break;
        }
        case K_M8: {
            uint32_t t[kR]; ld_m8(base + c.lane * 2, t);
#pragma unroll
            for (int r = 0; r < kR; r++) v[r] = t[r];
            break;
        }
        case K_STR:
#pragma unroll
            for (int r = 0; r < kR; r++)
                v[r] = (int64_t)(P.str_ptr[off] + (size_t)(c.row0 + row_in_tile(r, c.lane)) * P.str_w[off]);
            break;
        case K_IMM2: {
            const int64_t k2 = P.imm[off];
#pragma unroll
            for (int r = 0; r < kR; r++) v[r] = k2;
            break;
        }
        default:
#pragma unroll
            for (int r = 0; r < kR; r++) v[r] = imm;
            break;
    }
}
__device__ __forceinline__ void fetch_vref(const KParams& P, const WarpCtx& c, VRef vr, int64_t (&v)[kR]) {
    fetch(P, c, vr.kind, vr.slot & 1, vr.kind == K_STR ? (uint32_t)vr.off16 : ((uint32_t)vr.off16 << 4),
          vr.kind == K_IMM ? P.imm[vr.off16] : 0, v);
}

// one tuple of a sink value
__device__ __forceinline__ int64_t ld_row(const KParams& P, const WarpCtx& c, VRef vr, int r) {
    const int row = row_in_tile(r, c.lane);
    const uint32_t b = ((vr.slot & 1) ? c.wbase : c.stage) + ((uint32_t)vr.off16 << 4);
    switch (vr.kind) {
        case K_M64: return lds_b64(b + row * 8);
        case K_M32: return lds_s32(b + row * 4);
        case K_M8:  return lds_u8(b + row);
        case K_IMM: return P.imm[vr.off16];
        case K_STR: return (int64_t)(P.str_ptr[vr.off16] + (size_t)(c.row0 + row) * P.str_w[vr.off16]);
        default:    return 0;
    }
}

// packed group key: every key is a bit field of one word. In the 32-bit form (P.key32) every
// field is wide enough for its value by construction (pack_group_key sizes it from the value bounds
// or the physical width), so no masking is needed.
template <class Sp>
__device__ __forceinline__ void pack_keys32(const KParams& P, const WarpCtx& c, uint32_t (&k32)[kR]) {
#pragma unroll
    for (int r = 0; r < kR; r++) k32[r] = 0;
    for (int j = 0; j < Sp::nk(P); j++) {
        const VRef vr = Sp::key(P, j);
        const int sh = Sp::key_shift(P, j);
        const uint32_t base = ((vr.slot & 1) ? c.wbase : c.stage) + ((uint32_t)vr.off16 << 4);
        if (vr.kind == K_M8) {
            uint32_t t[kR];
            ld_m8(base + c.lane * 2, t);
            const uint32_t mul = 1u << sh;          // fields do not overlap: k32 + (t << sh) in one IMAD
#pragma unroll
            for (int r = 0; r < kR; r++) k32[r] = t[r] * mul + k32[r];
        } else if (vr.kind == K_M32) {
            int32_t t[kR];
            ld_m32(base + c.lane * 8, t);
#pragma unroll
            for (int r = 0; r < kR; r++) k32[r] |= (uint32_t)t[r] << sh;
        } else {
            int64_t kv[kR];
            fetch_vref(P, c, vr, kv);
#pragma unroll
            for (int r = 0; r < kR; r++) k32[r] |= (uint32_t)kv[r] << sh;
        }
    }
}
template <class Sp>
__device__ __forceinline__ void pack_keys(const KParams& P, const WarpCtx& c, uint64_t (&key)[kR]) {
    if (Sp::key32(P)) {
        uint32_t k32[kR];
        pack_keys32<Sp>(P, c, k32);
#pragma unroll
        for (int r = 0; r < kR; r++) key[r] = k32[r];
        return;
    }
#pragma unroll
    for (int r = 0; r < kR; r++) key[r] = 0;
    for (int j = 0; j < Sp::nk(P); j++) {
        int64_t kv[kR];
        fetch_vref(P, c, Sp::key(P, j), kv);
        const int sh = Sp::key_shift(P, j);
        const uint64_t mask = Sp::key_bits(P, j) >= 64 ? ~0ULL : ((1ULL << Sp::key_bits(P, j)) - 1);
#pragma unroll
        for (int r = 0; r < kR; r++) key[r] |= ((uint64_t)kv[r] & mask) << sh;
    }
}

// element i of a register array, and setting it: one compare-select per element keeps the array in
// registers, where a dynamic index would move it to local memory
template <typename T, int N>
__device__ __forceinline__ T reg_at(const T (&a)[N], int i) {
    T x = 0;
#pragma unroll
    for (int q = 0; q < N; q++) if (q == i) x = a[q];
    return x;
}
template <typename T, int N>
__device__ __forceinline__ void reg_set(T (&a)[N], int i, T x) {
#pragma unroll
    for (int q = 0; q < N; q++) if (q == i) a[q] = x;
}

// ---- low-cardinality global group table (packed key) -----------------------------------------
// The set test (U_GEN with D_INSET): which of the 8 tuples of a lane hold a value in the constant set S
// (rq_internal.h InSetHeader), as a bit mask. The set is read through the read-only path; it is small
// enough to stay in L2. Strings of tuples outside `valid` are not touched (they may lie past the column).
// The operand is a staged column or a slot read in its width, or a string column (encode_program refuses
// any other kind).
// Not inlined, like str_like: inside the interpreter switch it would change the register allocation of
// every kernel variant. It is an operation of the generic unit rather than a unit code of its own: a
// case of its own in the unit switch changed the dispatch of every other unit, and Q3 took 4 % longer.
// xa: shared address of the operand (staged column or slot); a string column is at sbase, sw bytes a row.
__device__ __noinline__ uint32_t inset_unit(uint32_t xa, uint32_t xkind, const unsigned char* sbase, uint32_t sw, uint32_t tile,
                                            int lane, const uint64_t* S, unsigned valid) {
    int64_t v[kR];
    if (xkind == K_STR) {
#pragma unroll
        for (int r = 0; r < kR; r++) v[r] = (int64_t)(sbase + ((size_t)tile * kTile + row_in_tile(r, lane)) * sw);
    } else if (xkind == K_M64) {
        ld_m64(xa + lane * 16, v);
    } else if (xkind == K_M32) {
        int32_t t[kR]; ld_m32(xa + lane * 8, t);
#pragma unroll
        for (int r = 0; r < kR; r++) v[r] = t[r];
    } else {
        uint32_t t[kR]; ld_m8(xa + lane * 2, t);
#pragma unroll
        for (int r = 0; r < kR; r++) v[r] = t[r];
    }
    const uint64_t form = __ldg(S), a = __ldg(S + 1), b = __ldg(S + 2);
    uint32_t hit = 0;
    if (form == IS_BITMAP) {
        const uint32_t* bits = reinterpret_cast<const uint32_t*>(S + 4);
#pragma unroll
        for (int r = 0; r < kR; r++) {
            const uint64_t d = (uint64_t)v[r] - a;
            if (d <= b) hit |= ((__ldg(bits + (d >> 5)) >> (d & 31)) & 1u) << r;
        }
    } else if (form == IS_SORTED) {
        // branchless binary search; the 8 searches of a lane advance together, so their loads are in
        // flight at the same time
        const int64_t* x = reinterpret_cast<const int64_t*>(S + 4);
        uint32_t base[kR];
#pragma unroll
        for (int r = 0; r < kR; r++) base[r] = 0;
        for (uint32_t len = (uint32_t)a; len > 1;) {
            const uint32_t half = len >> 1;
#pragma unroll
            for (int r = 0; r < kR; r++) base[r] = __ldg(x + base[r] + half) <= v[r] ? base[r] + half : base[r];
            len -= half;
        }
        if (a != 0) {
#pragma unroll
            for (int r = 0; r < kR; r++) hit |= (__ldg(x + base[r]) == v[r] ? 1u : 0u) << r;
        }
    } else {
        const bool chr = form == IS_CHAR;
        const char* blk = reinterpret_cast<const char*>(S);
#pragma unroll 1
        for (int r = 0; r < kR; r++) {
            if (!((valid >> r) & 1)) continue;
            const char* s = reinterpret_cast<const char*>(reg_at(v, r));
            const uint64_t h = inset_str_hash(s, chr);
            for (uint64_t i = h & a;; i = (i + 1) & a) {
                const uint64_t off = __ldg(S + 4 + 2 * i + 1);
                if (off == 0) break;
                if (__ldg(S + 4 + 2 * i) == h && (chr ? str_eq_char(s, blk + off) : str_eq_varchar(s, blk + off))) { hit |= 1u << r; break; }
            }
        }
    }
    return hit;
}

__device__ __forceinline__ int group_table_slot(const KParams& P, uint64_t key) {
    uint64_t hh = mix64(key ^ 0x9E3779B97F4A7C15ULL);
    uint32_t i = (uint32_t)(hh & (kGroupTableCap - 1));
    for (int tries = 0; tries < kGroupTableCap; tries++) {
        uint32_t st = atomicCAS(&P.g_state[i], 0u, 1u);
        if (st == 0u) {
            ((volatile int64_t*)P.g_keys)[i] = (int64_t)key;
            __threadfence();
            atomicExch(&P.g_state[i], 2u);
            return (int)i;
        }
        while (st == 1u) st = *(volatile uint32_t*)&P.g_state[i];
        __threadfence();
        if ((uint64_t)((volatile int64_t*)P.g_keys)[i] == key) return (int)i;
        i = (i + 1) & (kGroupTableCap - 1);
    }
    return -1;
}
// the same for a whole warp: lane 0 looks the key up (with nk = 0 grouping keys, the one key 0) and
// raises the overflow flag when the table is full; every lane gets the slot (-1: full)
__device__ __forceinline__ int warp_group_slot(const KParams& P, int nk, uint64_t key, int lane) {
    int slot = -1;
    if (lane == 0) {
        slot = group_table_slot(P, nk == 0 ? 0ULL : key);
        if (slot < 0) *P.overflow = 1;
    }
    return __shfl_sync(kFull, slot, 0);
}

__device__ __forceinline__ int64_t warp_reduce(int64_t v, int kind) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const int64_t w = __shfl_xor_sync(kFull, v, o);
        if (kind == RQ_AGG_MIN) v = w < v ? w : v;
        else if (kind == RQ_AGG_MAX) v = w > v ? w : v;
        else v = (int64_t)((uint64_t)v + (uint64_t)w);
    }
    return v;
}

__device__ __forceinline__ void group_table_add(const KParams& P, int slot, int a, int kind, int64_t v) {
    int64_t* dst = &P.g_acc[(size_t)slot * kMaxAggs + a];
    if (kind == RQ_AGG_MIN) atomicMin((long long*)dst, (long long)v);
    else if (kind == RQ_AGG_MAX) atomicMax((long long*)dst, (long long)v);
    else atomicAdd((unsigned long long*)dst, (unsigned long long)v);
}

// adds tuple r to aggregate a, whose word is acc[a] (hash aggregation and groupjoin entries)
template <class Sp>
__device__ __forceinline__ void atomic_agg(const KParams& P, const WarpCtx& c, uint64_t* acc, int a, int r) {
    const int kind = Sp::agg_kind(P, a);
    if (kind == RQ_AGG_COUNT) { atomicAdd((unsigned long long*)&acc[a], 1ULL); return; }
    const int64_t v = ld_row(P, c, Sp::agg_src(P, a), r);
    if (kind == RQ_AGG_SUM) atomicAdd((unsigned long long*)&acc[a], (unsigned long long)v);
    else if (kind == RQ_AGG_MIN) atomicMin((long long*)&acc[a], (long long)v);
    else atomicMax((long long*)&acc[a], (long long)v);
}

// group match: the key of the first unmatched tuple (bit of `unk`) of the lowest lane that has one,
// on every lane
__device__ __forceinline__ uint64_t leader_key(unsigned unk, const uint64_t (&key)[kR]) {
    const unsigned ball = __ballot_sync(kFull, unk != 0);
    const int leader = __ffs(ball) - 1;
    const uint64_t lk = reg_at(key, __ffs(unk) - 1);
    return __shfl_sync(kFull, lk, leader);
}

// a probe match of the tuple at `row`: the entry's payload words go to their value slots and, in the
// late variant, the entry reference `ref` to the probe's reference slot
template <bool LATE, class Sp>
__device__ __forceinline__ void put_match(const KParams& P, const DProbe& pr, int p, uint32_t wbase, int row,
                                          const uint64_t* ent, int64_t ref) {
    for (int q = 0; q < Sp::pr_n_out(pr, p); q++)
        if (Sp::pr_out_slot(pr, p, q) != 0xff)
            sts_b64(wbase + Sp::slots_rel(P) + Sp::pr_out_slot(pr, p, q) * (kTile * 8) + row * 8, (int64_t)ent[Sp::pr_pay_word(pr, p, q)]);
    if constexpr (LATE) {
        if (P.late_ref_slot[p] != 0xff)
            sts_b64(wbase + P.slots_rel + P.late_ref_slot[p] * (kTile * 8) + row * 8, ref);
    }
}

// ------------------------------------------------------------------------------------------
// the scan kernel
// ------------------------------------------------------------------------------------------
extern __shared__ __align__(128) unsigned char rq_smem[];

#define RQ_EX_ADD(x, y)  ((int64_t)((uint64_t)(x) + (uint64_t)(y)))
#define RQ_EX_SUB(x, y)  ((int64_t)((uint64_t)(x) - (uint64_t)(y)))
#define RQ_EX_RSUB(x, y) ((int64_t)((uint64_t)(y) - (uint64_t)(x)))
#define RQ_EX_MUL(x, y)  ((int64_t)((uint64_t)(x) * (uint64_t)(y)))
#define RQ_EX_AND(x, y)  ((x) & (y))
#define RQ_EX_OR(x, y)   ((x) | (y))
#define RQ_EX_LT(x, y)   ((int64_t)((x) < (y)))
#define RQ_EX_LE(x, y)   ((int64_t)((x) <= (y)))
#define RQ_EX_GT(x, y)   ((int64_t)((x) > (y)))
#define RQ_EX_GE(x, y)   ((int64_t)((x) >= (y)))
#define RQ_EX_EQ(x, y)   ((int64_t)((x) == (y)))
#define RQ_EX_NE(x, y)   ((int64_t)((x) != (y)))

// Nested-loops join source (CROSS, instantiated with GR = 0 only): the pairs of two relations are
// never materialized. Tile t holds pairs [256t, 256t + 256); pair p is (outer row p / n_inner, inner
// row p % n_inner). The host makes the smaller relation the inner one: consecutive pairs sweep the
// inner relation while the outer row changes once every n_inner pairs, so the columns read again and
// again are the smaller ones (at most 2^20 rows under the 2^40-pair limit: 8 MB per column, L2
// resident), and the outer row of a tile is one broadcast load. The warp stages a tile itself with
// plain loads at the offsets a bulk copy would use; there are no bulk copies and no mbarriers.
// Row counts are read on the device, clamped to each relation's capacity and to the pair count the
// host sized the launch for, so a wrong replay prediction cannot gather outside an allocation.
__device__ __forceinline__ int64_t cross_pairs(const KParams& P, uint64_t& n_inner) {
    int64_t n[2];
#pragma unroll
    for (int k = 0; k < 2; k++) {
        n[k] = *P.cross_rows[k];
        n[k] = n[k] < 0 ? 0 : (n[k] > P.cross_cap[k] ? P.cross_cap[k] : n[k]);
    }
    n_inner = (uint64_t)n[1];
    if (n[0] == 0 || n[1] == 0) return 0;
    return n[1] > P.n_rows / n[0] ? P.n_rows : n[0] * n[1];
}

// Stages the pairs [row0, row0 + 256) of a cross source into the stage at c.stage. Pairs at or past
// n_rows read nothing and stage zeros.
__device__ __forceinline__ void cross_stage(const KParams& P, const WarpCtx& c, int64_t n_rows, uint64_t n_inner) {
    // one division per tile; a tuple's pair is at most 255 past the tile's first one
    const uint64_t p0 = (uint64_t)c.row0;
    const uint64_t o0 = p0 / n_inner, i0 = p0 - o0 * n_inner;
    uint64_t oi[kR], ii[kR];
    unsigned ok = 0;
#pragma unroll
    for (int r = 0; r < kR; r++) {
        const uint32_t row = (uint32_t)row_in_tile(r, c.lane);
        if (n_inner >= (uint64_t)kTile) {
            ii[r] = i0 + row; oi[r] = o0;
            if (ii[r] >= n_inner) { ii[r] -= n_inner; oi[r]++; }
        } else {    // an inner relation of fewer than 256 rows: one tile spans several outer rows
            const uint32_t d = (uint32_t)i0 + row, q = d / (uint32_t)n_inner;
            ii[r] = d - q * (uint32_t)n_inner; oi[r] = o0 + q;
        }
        if ((int64_t)(p0 + row) < n_rows) ok |= 1u << r;
    }
    for (int col = 0; col < P.n_cols; col++) {
        const int64_t* src = reinterpret_cast<const int64_t*>(P.col_ptr[col]);
        const bool inner = (P.cross_inner >> col) & 1u;
        int64_t v[kR];
#pragma unroll
        for (int r = 0; r < kR; r++) v[r] = ((ok >> r) & 1) ? __ldg(src + (inner ? ii[r] : oi[r])) : 0;
        st_m64(c.stage + P.col_off[col] + c.lane * 16, v);
    }
    __syncwarp();
}

// ---- staging ----------------------------------------------------------------------------------
// A warp's ring of S stages and the tiles it walks: first, first + stride, ... below t_end.
struct Ring {
    uint32_t bars;          // shared address of the warp's mbarriers, one per stage
    uint32_t wbase;         // shared address of the warp's region; stage s is at wbase + s * P.stage_bytes
    int      S;
    uint32_t stride, t_end;
    uint32_t guarded_tile;  // the partial last tile of a borrowed source (0xffffffff: none)
    uint64_t policy;        // L2 policy of the bulk copies
    int      n_runs;
    bool     hint;          // copy with the L2 policy
};

// One lane issues the bulk copies of all staged columns of a tile into stage s (uniform operands)
// after arming the stage's barrier with its byte count. The guarded tile is staged by plain loads.
template <class Sp>
__device__ __forceinline__ void issue_tile(const KParams& P, const Ring& g, uint32_t tile, int s) {
    if (tile == g.guarded_tile) return;
    if (elect_one()) {
        const uint32_t bar = g.bars + s * 8;
        const uint32_t dst0 = g.wbase + s * Sp::stage_bytes(P);
        const uint32_t t32 = tile;
        mbar_expect_tx_s(bar, Sp::stage_bytes(P));
        if (g.hint) {
            for (int c = 0; c < g.n_runs; c++)
                tma_bulk_g2s_hint(dst0 + Sp::run_off(P, c), P.run_ptr[c] + (size_t)t32 * Sp::run_stride(P, c), Sp::run_bytes(P, c), bar, g.policy);
        } else {
            for (int c = 0; c < g.n_runs; c++)
                tma_bulk_g2s_s(dst0 + Sp::run_off(P, c), P.run_ptr[c] + (size_t)t32 * Sp::run_stride(P, c), Sp::run_bytes(P, c), bar);
        }
    }
}

// Early exit on a full hash table: the bulk copies already issued into this warp's stages (tiles
// `tile` onwards, starting at stage s) must land before the CTA may exit (a pending cp.async.bulk
// into freed shared memory is undefined).
__device__ __forceinline__ void drain_ring(const Ring& g, uint32_t tile, int s, uint32_t phase) {
    int ds = s;
    uint32_t dphase = phase;
    for (int k = 0; k < g.S; k++) {
        const uint64_t t = (uint64_t)tile + (uint64_t)k * g.stride;
        if (t < g.t_end && (uint32_t)t != g.guarded_tile) mbar_wait_s(g.bars + ds * 8, dphase);
        if (++ds == g.S) { ds = 0; dphase ^= 1u; }
    }
}

// The tile at c.row0 is in stage s after this: the bulk copies have landed, or the guarded tail of
// a borrowed source was staged with plain loads (zeros past n_rows), or the warp staged the pairs of
// a cross source itself.
template <bool CROSS, class Sp>
__device__ __forceinline__ void stage_tile(const KParams& P, const WarpCtx& c, const Ring& g, uint32_t tile, int s,
                                           uint32_t phase, int64_t n_rows, uint64_t n_inner, int n_cols) {
    if constexpr (CROSS) {
        if (n_cols > 0) cross_stage(P, c, n_rows, n_inner);
    } else if (n_cols > 0) {
        if (tile == g.guarded_tile) {
            const int64_t rows = n_rows - c.row0;
            for (int col = 0; col < Sp::n_cols(P); col++) {
                const int w = Sp::col_w(P, col);
                const unsigned char* src = P.col_ptr[col] + (size_t)c.row0 * w;
                for (int i = c.lane; i < kTile * w; i += 32)
                    sts_u8(c.stage + Sp::col_off(P, col) + i, (i < rows * w) ? src[i] : 0u);
            }
            __syncwarp();
        } else {
            mbar_wait_s(g.bars + s * 8, phase);
        }
    }
}

// The tile this warp stages next is pulled into L2 while the current one is processed, so the bulk
// copy issued at the end of the tile is served from L2 (one stage per warp cannot hide the DRAM
// latency otherwise).
template <class Sp>
__device__ __forceinline__ void prefetch_next(const KParams& P, const Ring& g, uint32_t tile) {
    if (Sp::l2_prefetch(P) && elect_one()) {
        const uint64_t nt = (uint64_t)tile + (uint64_t)g.S * g.stride;
        if (nt < g.t_end && (uint32_t)nt != g.guarded_tile)
            for (int c = 0; c < g.n_runs; c++)
                tma_prefetch_l2(P.run_ptr[c] + (size_t)(uint32_t)nt * Sp::run_stride(P, c), Sp::run_bytes(P, c));
    }
}

// ---- sink pieces ------------------------------------------------------------------------------
// Kernel state changes only through reference parameters; NA / NK are the kernel's P.na / P.nk. The
// other sinks stay in the kernel body: moved into functions, even verbatim, each changed the SASS of
// the GR = 0 variants, and moving the probe unit that way cost Q3 8.5 % (profiles/r06_kernel_split_ab.txt).

// Groups a flush covers (register path and LOWAGG): the warp's dictionary entries, or with no GROUP BY
// key the one group if any lane aggregated a tuple.
__device__ __forceinline__ int flush_groups(int NK, int ngroups, unsigned seen) {
    int n = ngroups;
    if (NK == 0) n = __any_sync(kFull, seen != 0) ? 1 : 0;
    return n;
}

// Materialize (IMPL_EMIT): the output position of the lane's first surviving tuple. One atomic per warp
// tile, lanes take consecutive output ranges.
__device__ __forceinline__ int64_t emit_locate(const KParams& P, int lane, unsigned valid) {
    const int cnt = __popc(valid);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += t;
    }
    const int total = __shfl_sync(kFull, incl, 31);
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(P.out_count, (unsigned long long)total);
    base = __shfl_sync(kFull, base, 0);
    return (int64_t)base + (incl - cnt);
}

// Materialize (IMPL_EMIT). `valid` is read only.
template <class Sp>
__device__ __forceinline__ void sink_emit(const KParams& P, const WarpCtx& c, unsigned valid) {
    int64_t pos = emit_locate(P, c.lane, valid);
    // only the surviving tuples are visited (a selective pass leaves a few per warp tile)
    for (unsigned todo = valid; todo; todo &= todo - 1) {
        const int r = __ffs(todo) - 1;
        if (pos < P.out_cap)
            for (int k = 0; k < Sp::n_out(P); k++) P.out_col[k][pos] = ld_row(P, c, Sp::out(P, k), r);
        pos++;
    }
}

// One round of the round form (ROUNDS): the sink values [v0, v1) of the surviving tuples go to their
// output columns from `pos`, the position emit_locate found for the lane before the first round.
__device__ __forceinline__ void emit_put(const KParams& P, const WarpCtx& c, unsigned valid, int64_t pos, int v0, int v1) {
    for (unsigned todo = valid; todo; todo &= todo - 1) {
        const int r = __ffs(todo) - 1;
        if (pos < P.out_cap)
            for (int k = v0; k < v1; k++) P.rout_col[k][pos] = ld_row(P, c, P.rval[k], r);
        pos++;
    }
}

// End of the scan for IMPL_LOWAGG: warp-reduce the accumulators of the first n groups (at most P.G) and
// add them to the global group table.
template <class Sp, int ND>
__device__ __forceinline__ void flush_lowagg(const KParams& P, int lane, int NA, int NK, uint32_t sacc, int n,
                                             const uint64_t (&dk)[ND]) {
    if (n > Sp::G(P)) n = Sp::G(P);
    for (int e = 0; e < n; e++) {
        const int slot = warp_group_slot(P, NK, reg_at(dk, e), lane);
        for (int a = 0; a < NA; a++) {
            const int kind = Sp::agg_kind(P, a);
            const int64_t v = warp_reduce(lds_b64(sacc + ((e * NA + a) * 32 + lane) * 8), kind);
            if (lane == 0 && slot >= 0) group_table_add(P, slot, a, kind, v);
        }
    }
}

// LATE (instantiated with GR = 0 only): late materialization. The tile's row (pair) indices go to
// the slot P.late_row_rel before the program runs, and a probe writes the reference of its matched
// entry to slot P.late_ref_slot[p]; the materialize sink then writes these references as columns of
// a record that rq_late_gather resolves into values.
// ROUNDS (instantiated with GR = 0 and LATE only): sink rounds of a materialize (KParams::n_rounds). Per
// tile the prefix units run, the output positions are located once, then every round runs its units and
// stores its values, so the value slots bound one round instead of the whole sink.
// The spec the kernel reads its host-known fields through: GenericSpec (read from P) in the library, a
// FixedSpec in a run-time specialization (jit.h), which defines RQ_SCAN_SPEC before including this file.
// (A macro rather than a template parameter or a wrapper around the body: either would change the
// ahead-of-time kernels - their names, or their code, since the body would then be compiled as a
// function of its own before being inlined.)
#ifndef RQ_SCAN_SPEC
#define RQ_SCAN_SPEC GenericSpec
#endif
template <int GR, bool CROSS = false, bool LATE = false, bool ROUNDS = false>
__global__ void __launch_bounds__(kMaxWarps * 32, 1)
rq_scan_kernel(const __grid_constant__ KParams P) {
    using Sp = RQ_SCAN_SPEC;
    static_assert(!CROSS || GR == 0, "the cross-source variant has the generic sinks only");
    static_assert(!LATE || GR == 0, "the late variant has the generic sinks only");
    static_assert(!ROUNDS || (GR == 0 && !CROSS && LATE), "the round variant is the late one with rounds");
    constexpr int NG = GR > 0 ? GR : 1;                 // register groups
    constexpr int ND = GR > 0 ? GR : kLowCardMaxGroups; // dictionary entries
    // lane / warp-region base are used everywhere; they are made opaque so that the compiler keeps
    // them in registers instead of re-deriving them from S2R + parameter loads under register
    // pressure (S2R has a long fixed latency and showed up as 'wait' stalls all over the tile loop)
    int lane = threadIdx.x & 31;
    // The warp index is read through a lane-0 shuffle: the compiler then knows it is warp-uniform,
    // so the tile counter, stage index and every TMA operand live in uniform registers and a bulk
    // copy is issued straight from them (a per-lane address would be serialised by an
    // elect / R2UR loop per copy - 18 instructions per tuple in the first version of this kernel).
    const int warp = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);
    const int W = blockDim.x >> 5;
    const int S = Sp::stages(P);

    const uint32_t smem0 = smem_u32(rq_smem);
    const uint32_t bars = smem0 + warp * (kMaxStages * 8);
    const uint32_t wbase = smem0 + Sp::warp_off(P) + warp * Sp::warp_bytes(P);
    asm volatile("" : "+r"(lane));
    const uint32_t sacc = wbase + Sp::acc_rel(P);            // GR == 0 low-card path: [g][a][lane] int64

    int64_t n_rows = P.n_rows;
    if (P.n_rows_ptr) { n_rows = *P.n_rows_ptr; if (n_rows > P.n_rows_cap) n_rows = P.n_rows_cap; }
    uint64_t n_inner = 0;
    if constexpr (CROSS) n_rows = cross_pairs(P, n_inner);
    // tile indices are 32-bit (2^32 tiles = 10^12 rows): cheap to keep or recompute under register pressure
    const uint32_t n_tiles = (uint32_t)((n_rows + kTile - 1) / kTile);
    // a launch may be restricted to the tiles [tile_range[0], tile_range[1]) of the source: the row
    // range a selection on a sorted column can match at all (zone skipping), or one rank's share of a
    // replicated build table (engine_exec.inl "tile ranges")
    // (not in the 4-group register kernel: it has no register to spare - measured, the extra live value
    // cost Q1 2 % - and the host never hands it a range)
    uint32_t t_end = n_tiles, t_begin = 0;
    if (GR != 4 && P.tile_range) {
        t_begin = min(P.tile_range[0], n_tiles);
        t_end = max(min(P.tile_range[1], n_tiles), t_begin);
        // (read through a lane-0 shuffle so that the compiler keeps the loop bounds in uniform registers,
        // like the parameter-derived tile count they replace)
        t_begin = __shfl_sync(kFull, t_begin, 0);
        t_end = __shfl_sync(kFull, t_end, 0);
    }
    const uint32_t stride = gridDim.x * W;
    const uint32_t first = t_begin + blockIdx.x * W + warp;
    const int NA = Sp::na(P), NK = Sp::nk(P);
    const int sink = Sp::sink(P);

    // the program, decoded on the host, is copied to shared memory once per CTA
    const uint32_t prog = smem0 + Sp::prog_off(P);
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(P.insn);
        for (int i = threadIdx.x; i < Sp::n_insn(P) * 8; i += blockDim.x) sts_b32(prog + i * 4, src[i]);
    }
    if (!CROSS && lane == 0) {
        for (int s = 0; s < S; s++) mbar_init_s(bars + s * 8, 1);
        fence_mbar_init();
    }
    __syncthreads();
    // accumulators of the register path: per group 2 x kNAR 32-bit registers (an aggregate owns a
    // pair: one or two 32-bit piece sums, or one 64-bit sum / min / max) and a tuple counter
    uint32_t racc[NG][2 * kNAR];
    uint32_t rcnt[NG];
    uint64_t dk[ND];
    int ngroups = 0;
    unsigned seen = 0;     // (no GROUP BY) did this lane aggregate at least one tuple
    unsigned n_inserted = 0;   // hash sinks: entries this lane added to the table
    unsigned long long acct_before = 0, acct_added = 0;   // lane 0: table counter before / by the previous tile
    auto reset_racc = [&]() {
#pragma unroll
        for (int g = 0; g < NG; g++) {
            rcnt[g] = 0;
#pragma unroll
            for (int a = 0; a < kNAR; a++) {
                const uint64_t id = (uint64_t)agg_identity(a < NA ? Sp::agg_kind(P, a) : 0);
                racc[g][2 * a] = (uint32_t)id;
                racc[g][2 * a + 1] = (uint32_t)(id >> 32);
            }
        }
    };
    reset_racc();
#pragma unroll
    for (int e = 0; e < ND; e++) dk[e] = 0;
    // register path: warp-reduce every (group, aggregate) partial and add it to the global group table
    // (at the end of the scan, and every P.flush_tiles tiles so that 32-bit piece sums cannot wrap)
    auto flush_regs = [&]() {
        const int n = flush_groups(NK, ngroups, seen);
#pragma unroll
        for (int g = 0; g < NG; g++) {
            if (g >= n) continue;
            const int slot = warp_group_slot(P, NK, dk[g], lane);
#pragma unroll
            for (int a = 0; a < kNAR; a++) {
                if (a >= NA) continue;
                const int kind = Sp::agg_kind(P, a);
                const int mode = Sp::agg_mode(P, a);
                uint64_t part;
                if (kind == RQ_AGG_COUNT) part = rcnt[g];
                else if (kind == RQ_AGG_SUM && mode == AM_P1) part = racc[g][2 * a];
                else if (kind == RQ_AGG_SUM && mode == AM_P2) part = (uint64_t)racc[g][2 * a] + ((uint64_t)racc[g][2 * a + 1] << Sp::agg_shift(P, a));
                else part = (uint64_t)racc[g][2 * a] | ((uint64_t)racc[g][2 * a + 1] << 32);
                const int64_t v = warp_reduce((int64_t)part, kind);
                if (lane == 0 && slot >= 0) group_table_add(P, slot, a, kind, v);
            }
        }
        reset_racc();
    };
    // Mid-scan flush of the 32-bit accumulators only (piece sums and tuple counters), before any of
    // them can wrap: 16-bit halves are summed over the warp with REDUX, so a flush costs a few
    // hundred instructions per warp.
    auto warp_sum_u32 = [&](uint32_t x) -> uint64_t {
        const uint32_t lo = __reduce_add_sync(kFull, x & 0xffffu);
        const uint32_t hi = __reduce_add_sync(kFull, x >> 16);
        return (uint64_t)lo + ((uint64_t)hi << 16);
    };
    auto flush_small = [&]() {
        const int n = flush_groups(NK, ngroups, seen);
#pragma unroll
        for (int g = 0; g < NG; g++) {
            if (g >= n) continue;
            const int slot = warp_group_slot(P, NK, dk[g], lane);
#pragma unroll
            for (int a = 0; a < kNAR; a++) {
                if (a >= NA) continue;
                const int kind = Sp::agg_kind(P, a);
                const int mode = Sp::agg_mode(P, a);
                uint64_t part;
                if (kind == RQ_AGG_COUNT) part = warp_sum_u32(rcnt[g]);
                else if (kind == RQ_AGG_SUM && mode == AM_P1) { part = warp_sum_u32(racc[g][2 * a]); racc[g][2 * a] = 0; }
                else if (kind == RQ_AGG_SUM && mode == AM_P2) {
                    part = warp_sum_u32(racc[g][2 * a]) + (warp_sum_u32(racc[g][2 * a + 1]) << Sp::agg_shift(P, a));
                    racc[g][2 * a] = 0; racc[g][2 * a + 1] = 0;
                } else continue;
                if (lane == 0 && slot >= 0) group_table_add(P, slot, a, kind, (int64_t)part);
            }
            rcnt[g] = 0;
        }
    };
    int tiles_to_flush = P.flush_tiles;
    if (GR == 0 && sink == IMPL_LOWAGG) {
        for (int i = lane; i < Sp::G(P) * NA * 32; i += 32) sts_b64(sacc + i * 8, agg_identity(Sp::agg_kind(P, (i >> 5) % NA)));
    }
    __syncwarp();

    // a partial last tile of a borrowed (unpadded) source is staged with guarded plain loads;
    // scanned data is streamed once, so it is marked evict-first in L2
    const Ring ring{bars, wbase, S, stride, t_end,
                    (P.borrowed && ((uint32_t)n_rows & (kTile - 1)) != 0) ? n_tiles - 1 : 0xffffffffu,
                    l2_evict_first_policy(), Sp::n_runs(P), Sp::stream_hint(P) != 0};
    const int n_cols = Sp::n_cols(P);
    if (!CROSS && n_cols > 0) {
        for (int s = 0; s < S; s++)
            if ((uint64_t)first + (uint64_t)s * stride < t_end) issue_tile<Sp>(P, ring, first + s * stride, s);
    }

    int s = 0;
    uint32_t phase = 0;
    const bool hash_sink = (GR == 0) && (sink == IMPL_BUILD || sink == IMPL_HASHAGG);
    // (the tile counter cannot wrap: first + k * stride < n_tiles + stride <= 2^32 is checked on the host)
    for (uint32_t tile = first; tile < t_end; tile += stride) {
        // a full hash table makes the host regrow it and rerun: stop early
        if (hash_sink && *(volatile int32_t*)P.ht_full) {
            if (!CROSS && n_cols > 0) drain_ring(ring, tile, s, phase);
            break;
        }
        WarpCtx c;
        c.stage = wbase + s * Sp::stage_bytes(P);
        c.wbase = wbase;
        c.row0 = (int64_t)tile * (int64_t)kTile;
        c.lane = lane;

        stage_tile<CROSS, Sp>(P, c, ring, tile, s, phase, n_rows, n_inner, n_cols);
        if (!CROSS) prefetch_next<Sp>(P, ring, tile);

        unsigned valid = 0xffu;
        if (c.row0 + kTile > n_rows) {
            valid = 0;
#pragma unroll
            for (int r = 0; r < kR; r++)
                if (c.row0 + row_in_tile(r, lane) < n_rows) valid |= 1u << r;
        }
        if constexpr (LATE) {
            if (P.late_row) {
                int64_t rid[kR];
#pragma unroll
                for (int r = 0; r < kR; r++) rid[r] = c.row0 + row_in_tile(r, lane);
                st_m64(wbase + P.late_row_rel + lane * 16, rid);
                __syncwarp();
            }
        }

        // ---- 1. the program (ROUNDS: the prefix, then the units of each round after the locate
        //         or the previous round's stores) --------------------------------------------
        int64_t rpos = 0;
        int pc0 = 0;
        for (int rd = -1;; rd++) {     // the parts of the program: units [pc0, n_insn) of part rd
        const int n_insn = !ROUNDS ? Sp::n_insn(P) : rd < 0 ? P.prefix_end : (int)P.round_unit_end[rd];
        // (with a fixed spec the loop is unrolled and each unit's switch folds to its one case; a unit
        // that leaves no tuple ends the part: a jump to program_end there, pc = n_insn here)
#define RQ_STOP()                                                                             \
    do {                                                                                      \
        if constexpr (Sp::kFixed) goto program_end; else pc = n_insn;                         \
    } while (0)
#pragma unroll
        for (int pc = pc0; pc < n_insn; pc++) {
            const UInsn in = Sp::insn(P, prog, pc);
            const uint32_t xa = ((in.flags & UF_XSLOT) ? wbase : c.stage) + in.xrel;
            const uint32_t ya = ((in.flags & UF_YSLOT) ? wbase : c.stage) + in.yrel;
            // result handling, expanded inside every case so that t never crosses the switch
#define RQ_FINISH(t)                                                                          \
    do {                                                                                      \
        if (in.flags & UF_STORE) st_m64(wbase + in.dstrel + lane * 16, t);                    \
        if (in.flags & UF_FILTER) {                                                           \
            _Pragma("unroll") for (int r = 0; r < kR; r++)                                    \
                if ((t[r] & 0xff) == 0) valid &= ~(1u << r);                                  \
            if (!__any_sync(kFull, valid != 0)) RQ_STOP();                                    \
        }                                                                                     \
    } while (0)

            switch (in.code) {
#define RQ_CASES(N)                                                                        \
    case U_##N##_MM: {                                                                     \
        int64_t a[kR], b[kR], t[kR];                                                       \
        ld_m64(xa + lane * 16, a); ld_m64(ya + lane * 16, b);                              \
        _Pragma("unroll") for (int r = 0; r < kR; r++) t[r] = RQ_EX_##N(a[r], b[r]);       \
        RQ_FINISH(t);                                                                      \
        break;                                                                             \
    }                                                                                      \
    case U_##N##_MI: {                                                                     \
        int64_t a[kR], t[kR];                                                              \
        ld_m64(xa + lane * 16, a);                                                         \
        const int64_t y = in.imm;                                                          \
        _Pragma("unroll") for (int r = 0; r < kR; r++) t[r] = RQ_EX_##N(a[r], y);          \
        RQ_FINISH(t);                                                                      \
        break;                                                                             \
    }
                RQ_BINOPS(RQ_CASES)
#undef RQ_CASES

#define RQ_MULI(CODE, EXPR)                                                                \
    case CODE: {                                                                           \
        int64_t a[kR], b[kR], t[kR];                                                       \
        ld_m64(xa + lane * 16, a); ld_m64(ya + lane * 16, b);                              \
        const uint64_t k = (uint64_t)in.imm;                                               \
        _Pragma("unroll") for (int r = 0; r < kR; r++) {                                   \
            const uint64_t x = (uint64_t)a[r];                                             \
            t[r] = (int64_t)((EXPR) * (uint64_t)b[r]);                                     \
        }                                                                                  \
        RQ_FINISH(t);                                                                      \
        break;                                                                             \
    }
                RQ_MULI(U_MULADDI, x + k)
                RQ_MULI(U_MULSUBI, x - k)
                RQ_MULI(U_MULRSUBI, k - x)
#undef RQ_MULI
#define RQ_MULI32(CODE, EXPR)                                                              \
    case CODE: {                                                                           \
        int64_t a[kR], b[kR], t[kR];                                                       \
        ld_m64(xa + lane * 16, a); ld_m64(ya + lane * 16, b);                              \
        const uint32_t k = (uint32_t)in.imm;                                               \
        _Pragma("unroll") for (int r = 0; r < kR; r++) {                                   \
            const uint32_t x = (uint32_t)a[r];                                             \
            t[r] = (int64_t)((uint64_t)(uint32_t)(EXPR) * (uint64_t)(uint32_t)b[r]);       \
        }                                                                                  \
        RQ_FINISH(t);                                                                      \
        break;                                                                             \
    }
                RQ_MULI32(U_MULADDI32, x + k)
                RQ_MULI32(U_MULSUBI32, x - k)
                RQ_MULI32(U_MULRSUBI32, k - x)
                RQ_MULI32(U_MUL32_MM, ((void)k, x))
#undef RQ_MULI32

                case U_GEN: {
                    int64_t t[kR], b[kR];
                    fetch(P, c, in.xkind, in.flags & UF_XSLOT, in.xrel, in.imm, t);
                    if (in.gop != D_LD) fetch(P, c, in.ykind, in.flags & UF_YSLOT, in.yrel, in.imm, b);
                    switch (in.gop) {
#define RQ_GBIN(D, N) case D: _Pragma("unroll") for (int r = 0; r < kR; r++) t[r] = RQ_EX_##N(t[r], b[r]); break;
                        RQ_GBIN(D_ADD, ADD) RQ_GBIN(D_SUB, SUB) RQ_GBIN(D_RSUB, RSUB) RQ_GBIN(D_MUL, MUL)
                        RQ_GBIN(D_AND, AND) RQ_GBIN(D_OR, OR) RQ_GBIN(D_LT, LT) RQ_GBIN(D_LE, LE)
                        RQ_GBIN(D_GT, GT) RQ_GBIN(D_GE, GE) RQ_GBIN(D_EQ, EQ) RQ_GBIN(D_NE, NE)
#undef RQ_GBIN
                        case D_DIV:
#pragma unroll
                            for (int r = 0; r < kR; r++)
                                t[r] = ((valid >> r) & 1) ? div_trunc(t[r], b[r], P.err) : 0;
                            break;
                        case D_RDIV:
#pragma unroll
                            for (int r = 0; r < kR; r++)
                                t[r] = ((valid >> r) & 1) ? div_trunc(b[r], t[r], P.err) : 0;
                            break;
#define RQ_STRBIN(D, EXPR)                                                       \
    case D:                                                                      \
        _Pragma("unroll") for (int r = 0; r < kR; r++) {                         \
            const char* x = reinterpret_cast<const char*>(t[r]);                 \
            const char* y = reinterpret_cast<const char*>(b[r]);                 \
            t[r] = ((valid >> r) & 1) ? (EXPR) : 0;                              \
        }                                                                        \
        break;
                        RQ_STRBIN(D_EQC, str_eq_char(x, y))
                        RQ_STRBIN(D_EQV, str_eq_varchar(x, y))
                        RQ_STRBIN(D_NEC, 1 - str_eq_char(x, y))
                        RQ_STRBIN(D_NEV, 1 - str_eq_varchar(x, y))
                        RQ_STRBIN(D_LIKE, str_like(x, y))
                        RQ_STRBIN(D_RLIKE, str_like(y, x))
#undef RQ_STRBIN
                        case D_SEL: {
                            // t = (x & 0xff) ? y : z     (one WHEN/THEN arm of emitCase :720-754)
                            int64_t e[kR];
                            fetch(P, c, in.zkind, in.flags & UF_ZSLOT, in.zrel,
                                  in.zkind == K_IMM ? P.imm[in.zrel] : 0, e);
#pragma unroll
                            for (int r = 0; r < kR; r++) t[r] = (t[r] & 0xff) ? b[r] : e[r];
                            break;
                        }
                        case D_INSET: {   // x IN (constants): one membership test for the whole OR tree
                            const bool str = in.xkind == K_STR;
                            const uint32_t hit = inset_unit(xa, in.xkind, str ? P.str_ptr[in.xrel] : nullptr, str ? P.str_w[in.xrel] : 0,
                                                            tile, lane, reinterpret_cast<const uint64_t*>(in.imm), valid);
#pragma unroll
                            for (int r = 0; r < kR; r++) t[r] = (hit >> r) & 1;
                            break;
                        }
                        default: break;   // D_LD: t = x
                    }
                    RQ_FINISH(t);
                    break;
                }

            // selection-fused compares: the 8 tuple tests are independent and combined by a tree,
            // so the mask update is not a serial chain
#define RQ_DROP(ok)                                                                        \
    do {                                                                                   \
        const unsigned f = (((ok[0] ? 0u : 1u) | (ok[1] ? 0u : 2u)) | ((ok[2] ? 0u : 4u) | (ok[3] ? 0u : 8u))) |       \
                           (((ok[4] ? 0u : 16u) | (ok[5] ? 0u : 32u)) | ((ok[6] ? 0u : 64u) | (ok[7] ? 0u : 128u)));   \
        valid &= ~f;                                                                       \
        if (!__any_sync(kFull, valid != 0)) RQ_STOP();                                     \
    } while (0)
#define RQ_FCMP(N, OP)                                                                     \
    case U_F##N##_M64: {                                                                   \
        int64_t b[kR]; ld_m64(xa + lane * 16, b);                                          \
        const int64_t y = in.imm;                                                          \
        bool ok[kR];                                                                       \
        _Pragma("unroll") for (int r = 0; r < kR; r++) ok[r] = (b[r] OP y);                \
        RQ_DROP(ok);                                                                       \
        break;                                                                             \
    }                                                                                      \
    case U_F##N##_M32: {                                                                   \
        int32_t b[kR]; ld_m32(xa + lane * 8, b);                                           \
        const int32_t y = (int32_t)in.imm;                                                 \
        bool ok[kR];                                                                       \
        _Pragma("unroll") for (int r = 0; r < kR; r++) ok[r] = (b[r] OP y);                \
        RQ_DROP(ok);                                                                       \
        break;                                                                             \
    }                                                                                      \
    case U_F##N##_M8: {                                                                    \
        uint32_t b[kR]; ld_m8(xa + lane * 2, b);                                           \
        const int32_t y = (int32_t)in.imm;                                                 \
        bool ok[kR];                                                                       \
        _Pragma("unroll") for (int r = 0; r < kR; r++) ok[r] = ((int32_t)b[r] OP y);       \
        RQ_DROP(ok);                                                                       \
        break;                                                                             \
    }
                RQ_FCMP(LT, <) RQ_FCMP(LE, <=) RQ_FCMP(GT, >) RQ_FCMP(GE, >=) RQ_FCMP(EQ, ==) RQ_FCMP(NE, !=)
#undef RQ_FCMP
                case U_FRANGE_M64: {      // imm <= x <= imm + span, one unsigned compare
                    int64_t b[kR]; ld_m64(xa + lane * 16, b);
                    const uint64_t lo = (uint64_t)in.imm, span = (uint64_t)in.yrel | ((uint64_t)in.zrel << 32);
                    bool ok[kR];
#pragma unroll
                    for (int r = 0; r < kR; r++) ok[r] = ((uint64_t)b[r] - lo) <= span;
                    RQ_DROP(ok);
                    break;
                }
                case U_FRANGE_M32: {
                    int32_t b[kR]; ld_m32(xa + lane * 8, b);
                    const uint32_t lo = (uint32_t)in.imm, span = in.yrel;
                    bool ok[kR];
#pragma unroll
                    for (int r = 0; r < kR; r++) ok[r] = ((uint32_t)b[r] - lo) <= span;
                    RQ_DROP(ok);
                    break;
                }
                case U_FRANGE_M8: {
                    uint32_t b[kR]; ld_m8(xa + lane * 2, b);
                    const uint32_t lo = (uint32_t)in.imm, span = in.yrel;
                    bool ok[kR];
#pragma unroll
                    for (int r = 0; r < kR; r++) ok[r] = (b[r] - lo) <= span;
                    RQ_DROP(ok);
                    break;
                }
#undef RQ_DROP

                case U_PROBE: {
                    if (GR > 0) { *P.err = 2; break; }     // never lowered for these kernels (host checks)
                    // hash-join probe (hashjoin.h:118-214): tuples without a match are dropped, the
                    // matching entry's payload words land in value slots. All 8 tuples of a lane
                    // are hashed and tested against the build side's Bloom filter first (one L2
                    // resident 32-bit word each, 8 loads in flight); only the survivors walk the
                    // hash table.
                    const DProbe& pr = P.probe[in.aux];
                    if (Sp::pr_fetch(pr, in.aux)) {
                        // second pass of a multi-match expansion: the entry was found (and the tuple
                        // multiplied) by the first pass, only the payload is read here
                        int64_t ei[kR];
                        fetch_vref(P, c, Sp::pr_key(pr, in.aux, 0), ei);
#pragma unroll 1
                        for (int r = 0; r < kR; r++) {
                            if (!((valid >> r) & 1)) continue;
                            const int64_t e = reg_at(ei, r);
                            put_match<LATE, Sp>(P, pr, in.aux, wbase, row_in_tile(r, lane), ht_entry(pr.ht, (uint64_t)e), e);
                        }
                        __syncwarp();
                        break;
                    }
                    if (Sp::pr_direct(pr, in.aux)) {
                        // direct-address build side: one bit test per tuple (all 8 words of a lane are
                        // fetched together), the payload of a hit is one more load; no walk, no compare
                        int64_t dk8[kR];
                        fetch_vref(P, c, Sp::pr_key(pr, in.aux, 0), dk8);
                        uint32_t w[kR];
#pragma unroll
                        for (int r = 0; r < kR; r++) {
                            const uint64_t idx = (uint64_t)dk8[r] - (uint64_t)pr.ht.dlo;
                            w[r] = (((valid >> r) & 1) && idx < pr.ht.dsize) ? pr.ht.dbits[idx >> 5] : 0u;
                        }
#pragma unroll
                        for (int r = 0; r < kR; r++) {
                            const uint64_t idx = (uint64_t)dk8[r] - (uint64_t)pr.ht.dlo;
                            if (!((w[r] >> (idx & 31)) & 1u)) valid &= ~(1u << r);
                        }
                        if (!Sp::pr_bloom_only(pr, in.aux)) {
                            if constexpr (LATE) {
                                if (P.late_ref_slot[in.aux] != 0xff) {
                                    const uint32_t dst = wbase + Sp::slots_rel(P) + P.late_ref_slot[in.aux] * (kTile * 8);
#pragma unroll
                                    for (int r = 0; r < kR; r++)
                                        sts_b64(dst + row_in_tile(r, lane) * 8, (int64_t)((uint64_t)dk8[r] - (uint64_t)pr.ht.dlo));
                                }
                            }
#pragma unroll 1
                            for (int q = 0; q < Sp::pr_n_out(pr, in.aux); q++) {
                                if (Sp::pr_out_slot(pr, in.aux, q) == 0xff) continue;
                                const int word = Sp::pr_pay_word(pr, in.aux, q) - 2;      // < 0: the payload repeats the join key
                                const uint32_t dst = wbase + Sp::slots_rel(P) + Sp::pr_out_slot(pr, in.aux, q) * (kTile * 8);
                                int64_t pv[kR];
#pragma unroll
                                for (int r = 0; r < kR; r++) {
                                    const uint64_t idx = (uint64_t)dk8[r] - (uint64_t)pr.ht.dlo;
                                    pv[r] = word < 0 ? dk8[r]
                                                     : (((valid >> r) & 1) ? (int64_t)pr.ht.darr[idx * pr.ht.dnv + word] : 0);
                                }
#pragma unroll
                                for (int r = 0; r < kR; r++) sts_b64(dst + row_in_tile(r, lane) * 8, pv[r]);
                            }
                            __syncwarp();
                        }
                        if (!__any_sync(kFull, valid != 0)) RQ_STOP();
                        break;
                    }
                    const uint64_t cap = pr.ht.cap_mask + 1;
                    const int pnk = Sp::pr_nk(pr, in.aux);
                    const bool k1 = pnk == 1 && Sp::pr_key_kind(pr, in.aux, 0) == 0;   // one integer key: the usual join
                    uint64_t h[kR];
                    int64_t kv[kR];
                    if (k1) {
                        fetch_vref(P, c, Sp::pr_key(pr, in.aux, 0), kv);
#pragma unroll
                        for (int r = 0; r < kR; r++) h[r] = hash_int(pr.ht, kv[r]);
                    } else {
#pragma unroll
                        for (int r = 0; r < kR; r++) { h[r] = 0; kv[r] = 0; }
#pragma unroll 1
                        for (int r = 0; r < kR; r++) {
                            if (!((valid >> r) & 1)) continue;
                            int64_t k[kMaxKeys];
                            for (int j = 0; j < pnk; j++) k[j] = ld_row(P, c, Sp::pr_key(pr, in.aux, j), r);
                            reg_set(h, r, hash_typed(k, pr.ht.key_kind, pnk));
                        }
                    }
                    if (Sp::pr_bloom(pr, in.aux)) {
                        uint32_t w[kR];
#pragma unroll
                        for (int r = 0; r < kR; r++)
                            w[r] = ((valid >> r) & 1) ? pr.ht.bloom[bloom_word(pr.ht, h[r])] : 0u;
#pragma unroll
                        for (int r = 0; r < kR; r++) {
                            const uint32_t bits = bloom_bits(pr.ht, h[r]);
                            if ((w[r] & bits) != bits) valid &= ~(1u << r);
                        }
                    }
                    if (Sp::pr_bloom_only(pr, in.aux)) {
                        // semi-join reduction pass of a split pipeline: survivors are materialized
                        // and probed for real by the second pass (engine_exec.inl split_at_probe)
                        if (!__any_sync(kFull, valid != 0)) RQ_STOP();
                        break;
                    }
                    if (k1) {
                        // The home-slot tags of all surviving tuples are fetched together (one memory
                        // round trip per lane instead of one per tuple); a walk continues per tuple
                        // only where the home slot holds another key.
                        uint64_t tag0[kR];
#pragma unroll
                        for (int r = 0; r < kR; r++)
                            tag0[r] = ((valid >> r) & 1) ? *ht_entry(pr.ht, h[r] >> pr.ht.shift) : 0ULL;
#pragma unroll
                        for (int r = 0; r < kR; r++) {
                            if (!((valid >> r) & 1)) continue;
                            const uint64_t tag = h[r] | 2ULL;
                            uint64_t i = h[r] >> pr.ht.shift;
                            uint64_t t = tag0[r];
                            int64_t found = -1;
                            unsigned matches = 0;
                            for (uint64_t tries = 0; tries < cap && t != 0ULL; tries++) {
                                if (t == tag && (int64_t)ht_entry(pr.ht, i)[1] == kv[r]) {
                                    if (found < 0) found = (int64_t)i;
                                    matches++;
                                    if (Sp::pr_single(pr, in.aux)) break;
                                }
                                i = (i + 1) & pr.ht.cap_mask;
                                t = *ht_entry(pr.ht, i);
                            }
                            if (found < 0) { valid &= ~(1u << r); continue; }
                            if (matches > 1) atomicAdd(pr.dup_counter, (unsigned long long)(matches - 1));
                            put_match<LATE, Sp>(P, pr, in.aux, wbase, row_in_tile(r, lane), ht_entry(pr.ht, (uint64_t)found), found);
                        }
                    } else {
                        unsigned todo = valid;
                        while (todo) {
                            const int r = __ffs(todo) - 1;
                            todo &= todo - 1;
                            const uint64_t hr = reg_at(h, r);
                            int64_t k[kMaxKeys];
                            for (int j = 0; j < pnk; j++) k[j] = ld_row(P, c, Sp::pr_key(pr, in.aux, j), r);
                            const uint64_t tag = hr | 2ULL;
                            uint64_t i = hr >> pr.ht.shift;
                            int64_t found = -1;
                            unsigned matches = 0;
                            for (uint64_t tries = 0; tries < cap; tries++) {
                                const uint64_t t = *ht_entry(pr.ht, i);
                                if (t == 0ULL) break;
                                if (t == tag && slot_keys_equal(pr.ht, i, k)) {
                                    if (found < 0) found = (int64_t)i;
                                    matches++;
                                    if (Sp::pr_single(pr, in.aux)) break;
                                }
                                i = (i + 1) & pr.ht.cap_mask;
                            }
                            if (found < 0) { valid &= ~(1u << r); continue; }
                            if (matches > 1) atomicAdd(pr.dup_counter, (unsigned long long)(matches - 1));
                            put_match<LATE, Sp>(P, pr, in.aux, wbase, row_in_tile(r, lane), ht_entry(pr.ht, (uint64_t)found), found);
                        }
                    }
                    __syncwarp();
                    if (!__any_sync(kFull, valid != 0)) RQ_STOP();
                    break;
                }
                default: break;
            }
#undef RQ_FINISH
        }
    program_end: __attribute__((unused));
#undef RQ_STOP
        // End of one part of the program. The other variants run the whole program as one part. ROUNDS:
        // the prefix (rd = -1) is followed by the locate and round rd by its stores, then the units of
        // round rd + 1 run. No unit after the prefix drops a tuple, so the positions located once hold
        // for every round.
        if constexpr (ROUNDS) {
            if (rd < 0) {
                if (!__any_sync(kFull, valid != 0)) break;      // every tuple dropped: no round runs
                rpos = emit_locate(P, lane, valid);
            } else {
                emit_put(P, c, valid, rpos, rd == 0 ? 0 : P.round_val_end[rd - 1], P.round_val_end[rd]);
            }
            if (rd + 1 == P.n_rounds) break;                    // the last round stored its values
            pc0 = n_insn;                                       // round rd + 1 starts where this part ended
        } else {
            break;
        }
        }   // (the parts of the program; the loop body above is not indented for them)

        // ---- 2. the sink --------------------------------------------------------------------
        if (!ROUNDS && __any_sync(kFull, valid != 0)) {
            if (GR > 0) {
                // register path: group match -> 0/1 multipliers -> accumulate
                uint32_t m[NG][kR];
                const unsigned nvalid = __popc(valid & 0xffu);
                if (NK == 0) {
                    seen |= valid;
#pragma unroll
                    for (int r = 0; r < kR; r++) m[0][r] = (valid >> r) & 1u;
#pragma unroll
                    for (int g = 1; g < NG; g++)
#pragma unroll
                        for (int r = 0; r < kR; r++) m[g][r] = 0;
                    rcnt[0] += nvalid;
                } else {
                    // packed 32-bit keys use at most 31 bits: all-ones marks a dropped tuple, all-ones
                    // minus one an unused dictionary entry, and neither equals a real key
                    uint64_t key[kR];
                    uint32_t k32[kR];
                    if (Sp::key32(P)) {
                        pack_keys32<Sp>(P, c, k32);
#pragma unroll
                        for (int r = 0; r < kR; r++) {
                            key[r] = k32[r];
                            k32[r] = (valid & (1u << r)) ? k32[r] : 0xffffffffu;
                        }
                    } else {
                        pack_keys<Sp>(P, c, key);
                    }
                    for (;;) {
                        uint32_t ct[NG];
                        if (Sp::key32(P)) {
#pragma unroll
                            for (int g = 0; g < NG; g++) {
                                const uint32_t d = g < ngroups ? (uint32_t)dk[g] : 0xfffffffeu;
#pragma unroll
                                for (int r = 0; r < kR; r++) m[g][r] = (k32[r] == d) ? 1u : 0u;
                            }
                        } else {
#pragma unroll
                            for (int g = 0; g < NG; g++) {
                                const bool act = g < ngroups;
#pragma unroll
                                for (int r = 0; r < kR; r++)
                                    m[g][r] = (act && key[r] == dk[g] && ((valid >> r) & 1)) ? 1u : 0u;
                            }
                        }
                        // tuples per group in this tile; a valid tuple that matched no dictionary
                        // entry shows up as a shortfall against the number of valid tuples
                        unsigned known = 0;
#pragma unroll
                        for (int g = 0; g < NG; g++) {
                            ct[g] = ((m[g][0] + m[g][1]) + (m[g][2] + m[g][3])) + ((m[g][4] + m[g][5]) + (m[g][6] + m[g][7]));
                            known += ct[g];
                        }
                        if (__all_sync(kFull, known == nvalid)) {
#pragma unroll
                            for (int g = 0; g < NG; g++) rcnt[g] += ct[g];
                            break;
                        }
                        // slow path (first tiles of a warp): the key of the first unmatched tuple of the
                        // lowest lane joins the dictionary, then the multipliers are computed again
                        unsigned unk = 0;
#pragma unroll
                        for (int r = 0; r < kR; r++) {
                            uint32_t any = 0;
#pragma unroll
                            for (int g = 0; g < NG; g++) any |= m[g][r];
                            if ((valid & (1u << r)) && any == 0) unk |= 1u << r;
                        }
                        const uint64_t lk = leader_key(unk, key);
                        if (ngroups >= NG) {
                            // more groups than this path tracks: the host reruns with the next
                            // implementation; the unmatched tuples are simply dropped here
                            if (lane == 0) *P.overflow = 1;
                            valid &= ~unk;
#pragma unroll
                            for (int g = 0; g < NG; g++) rcnt[g] += ct[g];
                            break;
                        }
                        reg_set(dk, ngroups, lk);
                        ngroups++;
                    }
                }
                // The aggregate loop is unrolled, so every accumulator is a fixed register. A tuple
                // value goes into the accumulator of every group through the 0/1 group multiplier.
                // sm_100a has no fused 64-bit multiply-add (IMAD.WIDE + IADD3 + IADD3.X), so the host
                // picks the cheapest exact form per aggregate from the value bounds (upload
                // statistics + interval arithmetic; the first three need value >= 0):
                //   AM_P1   value < 2^25: one 32-bit accumulator, one IMAD per (group, tuple)
                //   AM_W64  value < 2^32: 64-bit accumulator, IMAD.WIDE.U32 + 64-bit add
                //   AM_P2   value < 2^48: two 32-bit accumulators for the low / high piece
                //   AM_FULL any int64   : 64-bit accumulator, wide multiply of the low word plus the
                //                         high word's low product (wrap-around int64 sum)
                // 32-bit accumulators are flushed to the global group table before they can wrap
                // (every P.flush_tiles tiles, see below).
#pragma unroll
                for (int a = 0; a < kNAR; a++) {
                    // one descriptor word per aggregate (host: choose_agg_modes): bits 0-2 form
                    // (0 = nothing to do here: COUNT or unused), bit 3 = 64-bit operand in shared
                    // memory at (bit 4 ? warp region : stage) + (desc >> 8)
                    const uint32_t desc = Sp::agg_desc(P, a);
                    const int form = (int)(desc & 7u);
                    if (form == AF_NONE) continue;
                    int64_t v[kR];
                    if (desc & 8u) ld_m64(((desc & 16u) ? c.wbase : c.stage) + (desc >> 8) + lane * 16, v);
                    else fetch_vref(P, c, Sp::agg_src(P, a), v);
                    const int kind = form == AF_MIN ? RQ_AGG_MIN : RQ_AGG_MAX;
                    if (form == AF_P1) {
#pragma unroll
                        for (int r = 0; r < kR; r++)
#pragma unroll
                            for (int g = 0; g < NG; g++) racc[g][2 * a] += (uint32_t)v[r] * m[g][r];
                    } else if (form == AF_P2) {
                        const int sh = Sp::agg_shift(P, a);
                        const uint32_t lomask = (1u << sh) - 1u;
#pragma unroll
                        for (int r = 0; r < kR; r++) {
                            const uint32_t lo = (uint32_t)v[r] & lomask;
                            const uint32_t hi = (uint32_t)((uint64_t)v[r] >> sh);
#pragma unroll
                            for (int g = 0; g < NG; g++) {
                                racc[g][2 * a] += lo * m[g][r];
                                racc[g][2 * a + 1] += hi * m[g][r];
                            }
                        }
                    } else if (form == AF_W64) {
#pragma unroll
                        for (int g = 0; g < NG; g++) {
                            uint64_t acc = (uint64_t)racc[g][2 * a] | ((uint64_t)racc[g][2 * a + 1] << 32);
#pragma unroll
                            for (int r = 0; r < kR; r++) acc += (uint64_t)(uint32_t)v[r] * (uint64_t)m[g][r];
                            racc[g][2 * a] = (uint32_t)acc; racc[g][2 * a + 1] = (uint32_t)(acc >> 32);
                        }
                    } else if (form == AF_FULL) {
#pragma unroll
                        for (int g = 0; g < NG; g++) {
                            uint64_t acc = (uint64_t)racc[g][2 * a] | ((uint64_t)racc[g][2 * a + 1] << 32);
#pragma unroll
                            for (int r = 0; r < kR; r++) {
                                acc += (uint64_t)(uint32_t)v[r] * (uint64_t)m[g][r];
                                acc += (uint64_t)((uint32_t)((uint64_t)v[r] >> 32) * m[g][r]) << 32;
                            }
                            racc[g][2 * a] = (uint32_t)acc; racc[g][2 * a + 1] = (uint32_t)(acc >> 32);
                        }
                    } else {                              // MIN / MAX
#pragma unroll
                        for (int g = 0; g < NG; g++) {
                            int64_t best = (int64_t)((uint64_t)racc[g][2 * a] | ((uint64_t)racc[g][2 * a + 1] << 32));
#pragma unroll
                            for (int r = 0; r < kR; r++)
                                if (m[g][r] && (kind == RQ_AGG_MIN ? v[r] < best : v[r] > best)) best = v[r];
                            racc[g][2 * a] = (uint32_t)(uint64_t)best; racc[g][2 * a + 1] = (uint32_t)((uint64_t)best >> 32);
                        }
                    }
                }
            } else if (sink == IMPL_LOWAGG) {
                // lane-private shared-memory accumulators [g][a][lane]
                unsigned gid = 0;   // 4 bits per tuple
                if (NK == 0) {
                    seen |= valid;
                } else {
                    uint64_t key[kR];
                    pack_keys<Sp>(P, c, key);
                    unsigned unk = 0;
#pragma unroll
                    for (int r = 0; r < kR; r++) {
                        unsigned g = 15;
#pragma unroll
                        for (int e = 0; e < ND; e++)
                            if (e < ngroups && key[r] == dk[e]) g = e;
                        if (!((valid >> r) & 1)) g = 0;
                        else if (g == 15) { unk |= 1u << r; g = 0; }
                        gid |= g << (4 * r);
                    }
                    while (__any_sync(kFull, unk != 0)) {
                        const uint64_t lk = leader_key(unk, key);
                        if (ngroups >= Sp::G(P)) {
                            if (lane == 0) *P.overflow = 1;
                            unk = 0;
                            break;
                        }
                        reg_set(dk, ngroups, lk);
#pragma unroll
                        for (int r = 0; r < kR; r++) {
                            if (((unk >> r) & 1) && key[r] == lk) {
                                unk &= ~(1u << r);
                                gid |= (unsigned)ngroups << (4 * r);
                            }
                        }
                        ngroups++;
                    }
                }
                for (int a = 0; a < NA; a++) {
                    const int kind = Sp::agg_kind(P, a);
                    int64_t v[kR];
                    if (kind != RQ_AGG_COUNT) fetch_vref(P, c, Sp::agg_src(P, a), v);
                    const uint32_t base = sacc + (a * 32 + lane) * 8;
#pragma unroll
                    for (int r = 0; r < kR; r++) {
                        if ((valid >> r) & 1) {
                            const uint32_t p = base + ((gid >> (4 * r)) & 15) * NA * 256;
                            const int64_t cur = lds_b64(p);
                            int64_t nv;
                            if (kind == RQ_AGG_COUNT) nv = cur + 1;
                            else if (kind == RQ_AGG_SUM) nv = (int64_t)((uint64_t)cur + (uint64_t)v[r]);
                            else if (kind == RQ_AGG_MIN) nv = v[r] < cur ? v[r] : cur;
                            else nv = v[r] > cur ? v[r] : cur;
                            sts_b64(p, nv);
                        }
                    }
                }
            } else if (sink == IMPL_BUILD) {
                // hash-join build (hashjoin.h:226-256): every tuple claims its own entry.
                const int bnk = Sp::ht_nk(P);
                if (Sp::ht_direct(P)) {
                    // direct-address build: set the key's bit, store its payload words (plain stores)
                    int64_t bk[kR];
                    fetch_vref(P, c, Sp::key(P, 0), bk);
                    uint32_t was[kR];          // the 8 bit-set atomics of a lane are in flight together
#pragma unroll
                    for (int r = 0; r < kR; r++) {
                        const uint64_t idx = (uint64_t)bk[r] - (uint64_t)P.ht.dlo;
                        was[r] = 0;
                        if (((valid >> r) & 1) && idx < P.ht.dsize) was[r] = atomicOr(&P.ht.dbits[idx >> 5], 1u << (idx & 31));
                    }
#pragma unroll 1
                    for (int r = 0; r < kR; r++) {
                        if (!((valid >> r) & 1)) continue;
                        const uint64_t idx = (uint64_t)bk[r] - (uint64_t)P.ht.dlo;
                        if (idx >= P.ht.dsize) { *const_cast<int32_t*>(P.ht_full + kDupKeyFromHtFull) = 1; continue; }   // outside the proven domain
                        if (was[r] & (1u << (idx & 31))) *const_cast<int32_t*>(P.ht_full + kDupKeyFromHtFull) = 1;     // duplicate key: the host falls back to the hash form
                        for (int q = 0; q < Sp::n_out(P); q++) P.ht.darr[idx * P.ht.dnv + q] = (uint64_t)ld_row(P, c, Sp::out(P, q), r);
                        for (int a = 0; a < NA; a++) P.ht.darr[idx * P.ht.dnv + P.gj_acc_word + a] = (uint64_t)agg_identity(Sp::agg_kind(P, a));
                        n_inserted++;
                    }
                } else if (bnk == 1 && Sp::ht_key_kind(P, 0) == 0) {
                    // One integer key. The claims (atomicCAS on the home slot) of a lane's tuples
                    // are issued together: a dense tile costs one atomic round trip per lane; a
                    // tuple whose home slot is taken walks on alone.
                    int64_t bk[kR];
                    fetch_vref(P, c, Sp::key(P, 0), bk);
                    unsigned long long old[kR];
#pragma unroll
                    for (int r = 0; r < kR; r++) {
                        old[r] = 1ULL;
                        if ((valid >> r) & 1) {
                            const uint64_t hh = hash_int(P.ht, bk[r]);
                            old[r] = atomicCAS((unsigned long long*)ht_entry(P.ht, hh >> P.ht.shift), 0ULL,
                                               (unsigned long long)(hh | 2ULL));
                        }
                    }
#pragma unroll
                    for (int r = 0; r < kR; r++) {
                        if (!((valid >> r) & 1)) continue;
                        const uint64_t hh = hash_int(P.ht, bk[r]);
                        uint64_t slot = hh >> P.ht.shift;
                        if (old[r] != 0ULL) {
                            if (!ht_insert_dup_from(P.ht, hh, (slot + 1) & P.ht.cap_mask, &slot, P.ht_full)) { *P.ht_full = 1; continue; }
                        }
                        uint64_t* e = ht_entry(P.ht, slot);
                        e[1] = (uint64_t)bk[r];
                        for (int q = 0; q < Sp::n_out(P); q++) e[2 + q] = (uint64_t)ld_row(P, c, Sp::out(P, q), r);
                        if (P.ht.bloom != nullptr) atomicOr(&P.ht.bloom[bloom_word(P.ht, hh)], bloom_bits(P.ht, hh));
                        n_inserted++;
                    }
                } else {
#pragma unroll 1
                    for (int r = 0; r < kR; r++) {
                        if (!((valid >> r) & 1)) continue;
                        int64_t k[kMaxKeys];
                        for (int j = 0; j < bnk; j++) k[j] = ld_row(P, c, Sp::key(P, j), r);
                        const uint64_t hh = hash_keys(P.ht, k);
                        uint64_t slot;
                        if (!ht_insert_dup(P.ht, k, hh, &slot, P.ht_full)) { *P.ht_full = 1; continue; }
                        uint64_t* e = ht_entry(P.ht, slot);
                        for (int q = 0; q < Sp::n_out(P); q++) e[1 + bnk + q] = (uint64_t)ld_row(P, c, Sp::out(P, q), r);
                        if (P.ht.bloom != nullptr) atomicOr(&P.ht.bloom[bloom_word(P.ht, hh)], bloom_bits(P.ht, hh));
                        n_inserted++;
                    }
                }
            } else if (sink == IMPL_HASHAGG && Sp::ht_packed(P)) {
                // GROUP BY whose keys pack into one word (bit fields from the value bounds, < 64 bits):
                // the entry's first word IS the key (+1, 0 = empty), so claiming a slot and publishing its
                // key are one atomicCAS - no lock state, no fence, nobody ever waits. The home-slot claims
                // of a lane's 8 tuples are issued together; aggregates are fire-and-forget atomics.
                uint64_t key[kR];
                pack_keys<Sp>(P, c, key);
                unsigned long long old[kR];
#pragma unroll
                for (int r = 0; r < kR; r++) {
                    old[r] = 0;
                    if ((valid >> r) & 1) {
                        const uint64_t hh = mix64(key[r] + 0x9E3779B97F4A7C15ULL);
                        old[r] = atomicCAS((unsigned long long*)ht_entry(P.ht, hh >> P.ht.shift), 0ULL, (unsigned long long)(key[r] + 1));
                    }
                }
#pragma unroll 1
                for (int r = 0; r < kR; r++) {
                    if (!((valid >> r) & 1)) continue;
                    const unsigned long long want = (unsigned long long)(key[r] + 1);
                    const uint64_t hh = mix64(key[r] + 0x9E3779B97F4A7C15ULL);
                    uint64_t slot = hh >> P.ht.shift;
                    unsigned long long cur = old[r];
                    bool ok = true;
                    for (uint64_t tries = 1; cur != 0ULL && cur != want; tries++) {
                        slot = (slot + 1) & P.ht.cap_mask;
                        cur = atomicCAS((unsigned long long*)ht_entry(P.ht, slot), 0ULL, want);
                        if ((tries & (kFullCheckEvery - 1)) == 0 && (*(volatile int32_t*)P.ht_full || tries > P.ht.cap_mask)) { ok = false; break; }
                    }
                    if (!ok) { *P.ht_full = 1; continue; }
                    if (cur == 0ULL) n_inserted++;
                    uint64_t* acc = ht_entry(P.ht, slot) + 1;
                    for (int a = 0; a < NA; a++) atomic_agg<Sp>(P, c, acc, a, r);
                }
            } else if (sink == IMPL_HASHAGG) {
                for (unsigned todo = valid; todo; todo &= todo - 1) {
                    const int r = __ffs(todo) - 1;
                    int64_t k[kMaxKeys];
                    for (int j = 0; j < Sp::ht_nk(P); j++) k[j] = ld_row(P, c, Sp::key(P, j), r);
                    const uint64_t hh = hash_keys(P.ht, k);
                    uint64_t slot;
                    bool fresh = false;
                    if (!ht_find_or_insert(P.ht, k, hh, &slot, &fresh, P.ht_full)) { *P.ht_full = 1; continue; }
                    if (fresh) n_inserted++;
                    uint64_t* acc = ht_entry(P.ht, slot) + 1 + Sp::ht_nk(P);
                    for (int a = 0; a < NA; a++) atomic_agg<Sp>(P, c, acc, a, r);
                }
            } else if (sink == IMPL_GROUPJOIN) {
                // GROUP BY on the key of a direct-address join (engine_exec.inl groupjoin_probe): the
                // probe in front kept only tuples whose key has an entry, and each entry is exactly one
                // group. A tuple marks its entry touched and adds into the entry's accumulator words
                // with fire-and-forget atomics; the group's other keys stay in the entry until the
                // compaction reads them once per group.
                int64_t gk[kR];
                fetch_vref(P, c, Sp::key(P, 0), gk);
#pragma unroll 1
                for (int r = 0; r < kR; r++) {
                    if (!((valid >> r) & 1)) continue;
                    const uint64_t idx = (uint64_t)reg_at(gk, r) - (uint64_t)P.ht.dlo;
                    atomicOr(&P.gj_touched[idx >> 5], 1u << (idx & 31));
                    uint64_t* acc = P.ht.darr + idx * P.ht.dnv + P.gj_acc_word;
                    for (int a = 0; a < NA; a++) atomic_agg<Sp>(P, c, acc, a, r);
                }
            } else if (sink == IMPL_EMIT && Sp::expand_probe(P) >= 0) {
                // multi-match hash join (hashjoin.h:118-165): one output row per key-equal entry.
                // The probe unit in front only applied the Bloom filter; here every surviving tuple
                // walks its chain and emits (its values, entry index) once per match.
                const DProbe& pr = P.probe[Sp::expand_probe(P)];
                const uint64_t cap = pr.ht.cap_mask + 1;
                const int pnk = pr.ht.nk;
#pragma unroll 1
                for (int r = 0; r < kR; r++) {
                    if (!((valid >> r) & 1)) continue;
                    int64_t k[kMaxKeys];
                    for (int j = 0; j < pnk; j++) k[j] = ld_row(P, c, pr.key[j], r);
                    const uint64_t hr = hash_keys(pr.ht, k);
                    const uint64_t tag = hr | 2ULL;
                    uint64_t i = hr >> pr.ht.shift;
                    for (uint64_t tries = 0; tries < cap; tries++) {
                        const uint64_t t = *ht_entry(pr.ht, i);
                        if (t == 0ULL) break;
                        if (t == tag && slot_keys_equal(pr.ht, i, k)) {
                            const unsigned long long pos = atomicAdd(P.out_count, 1ULL);
                            if ((int64_t)pos < P.out_cap) {
                                for (int q = 0; q < Sp::n_out(P); q++) P.out_col[q][pos] = ld_row(P, c, Sp::out(P, q), r);
                                P.out_col[Sp::n_out(P)][pos] = (int64_t)i;
                            }
                            if (pr.single) break;
                        }
                        i = (i + 1) & pr.ht.cap_mask;
                    }
                }
            } else if (sink == IMPL_EMIT) {
                sink_emit<Sp>(P, c, valid);
            }
        }

        // hash sinks: the entries this warp added go to the table's counter tile by tile; crossing the
        // load limit raises the table-full flag (the host regrows and reruns)
        if (hash_sink) {
            unsigned tot = n_inserted;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(kFull, tot, o);
            // (the counter's old value is only looked at one tile later, so nobody waits for the atomic)
            if (lane == 0) {
                if (acct_before + acct_added > P.ht.limit) *P.ht_full = 1;
                acct_added = tot;
                acct_before = tot ? atomicAdd(P.ht_entries, (unsigned long long)tot) : 0ULL;
            }
            n_inserted = 0;
        }
        // everyone is done with stage s (and the slots) before it is refilled
        __syncwarp();
        if (!CROSS && n_cols > 0) {
            const uint64_t nt = (uint64_t)tile + (uint64_t)S * stride;
            if (nt < t_end) issue_tile<Sp>(P, ring, (uint32_t)nt, s);
        }
        if (++s == S) { s = 0; phase ^= 1u; }
        if (GR > 0 && P.flush_tiles > 0 && --tiles_to_flush == 0) {
            flush_small();
            tiles_to_flush = P.flush_tiles;
        }
    }

    // ---- flush the per-warp accumulators of the low-cardinality aggregate -------------------
    if (GR > 0 || sink == IMPL_LOWAGG) {
        __syncwarp();
        const int n = flush_groups(NK, ngroups, seen);
        if (GR > 0) flush_regs();
        else flush_lowagg<Sp>(P, lane, NA, NK, sacc, n, dk);
    }
}

#ifndef __CUDACC_RTC__     // (a run-time compiled specialization, jit.h, needs only the kernel body above)
// The instantiations of the scan kernel and the one a launch uses: gr is the number of register
// groups (0, 1 or 4); the cross-source, late and round variants exist for gr = 0 only and take precedence.
using ScanKernel = void (*)(KParams);
inline ScanKernel scan_kernel_for(int gr, bool cross, bool late, bool rounds) {
    if (rounds) return rq_scan_kernel<0, false, true, true>;
    if (late) return cross ? rq_scan_kernel<0, true, true> : rq_scan_kernel<0, false, true>;
    if (cross) return rq_scan_kernel<0, true>;
    return gr == 4 ? rq_scan_kernel<4> : gr == 1 ? rq_scan_kernel<1> : rq_scan_kernel<0>;
}

// ------------------------------------------------------------------------------------------
// small helper kernels
// ------------------------------------------------------------------------------------------
// reset the global group table: state 0, accumulators to their identities
struct AggKinds { uint8_t kind[kMaxAggs]; };
__global__ void rq_group_table_init(uint32_t* state, int64_t* acc, AggKinds kinds, int na) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < kGroupTableCap) {
        state[i] = 0;
        for (int a = 0; a < na; a++) acc[(size_t)i * kMaxAggs + a] = agg_identity(kinds.kind[a]);
    }
}

struct KeyUnpack {
    int32_t nk;
    uint8_t shift[kMaxKeys];
    uint8_t bits[kMaxKeys];
    uint8_t sign[kMaxKeys];    // sign-extend the field (INT/DATE/BIGINT/DECIMAL keys)
};

// group table -> dense int64 columns (keys unpacked first, then aggregates); order is
// unspecified, as in the reference where it is hash-slot order (aggregation.h:298-343)
struct ColPtrs { int64_t* p[kMaxOut]; };
__global__ void rq_group_table_compact(const uint32_t* state, const int64_t* keys,
                                       const int64_t* acc, KeyUnpack ku, int na,
                                       ColPtrs out_cols, int64_t* out_count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < kGroupTableCap && state[i] == 2u) {
        const long long pos = atomicAdd((unsigned long long*)out_count, 1ULL);
        const uint64_t k = (uint64_t)keys[i];
        for (int j = 0; j < ku.nk; j++) {
            const int b = ku.bits[j];
            uint64_t f = (b >= 64) ? k : ((k >> ku.shift[j]) & ((1ULL << b) - 1));
            if (ku.sign[j] && b < 64 && ((f >> (b - 1)) & 1)) f |= ~((1ULL << b) - 1);
            out_cols.p[j][pos] = (int64_t)f;
        }
        for (int a = 0; a < na; a++) out_cols.p[ku.nk + a][pos] = acc[(size_t)i * kMaxAggs + a];
    }
}

// address of row i of a column: plain arrays have tile_stride == kTile * width, tile-major tables
// the page size
__device__ __forceinline__ const unsigned char* col_row(const unsigned char* col, int width, int64_t tile_stride, int64_t i) {
    return col + (i / kTile) * tile_stride + (i % kTile) * width;
}

// a few host bytes -> device memory as kernel ARGUMENTS (no host buffer is read when the launch
// executes, so the launch can be recorded into a CUDA graph and replayed)
struct SmallBytes { unsigned char b[64]; };
__global__ void rq_store_bytes(unsigned char* dst, SmallBytes v, int n) {
    if ((int)threadIdx.x < n) dst[threadIdx.x] = v.b[threadIdx.x];
}

// is an integer column non-decreasing over the rows? *flag is cleared when a descent is found
__global__ void rq_col_sorted(const unsigned char* col, int width, int64_t tile_stride, int64_t n, int32_t* flag) {
    int seen = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i + 1 < n; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned char* p = col_row(col, width, tile_stride, i);
        const unsigned char* q = col_row(col, width, tile_stride, i + 1);
        int64_t a, b;
        if (width == 8) { a = *reinterpret_cast<const int64_t*>(p); b = *reinterpret_cast<const int64_t*>(q); }
        else if (width == 4) { a = *reinterpret_cast<const int32_t*>(p); b = *reinterpret_cast<const int32_t*>(q); }
        else { a = *p; b = *q; }
        // one writer is enough, and nobody needs to look further once the answer is known (an unsorted
        // column would otherwise make every thread hammer the same word)
        if (a > b) { *flag = 0; return; }
        if ((++seen & 15) == 0 && *(volatile int32_t*)flag == 0) return;
    }
}

// tiles of a non-decreasing column that can hold a value in [lo, hi]: out = [first tile, last tile + 1),
// intersected with the range already there (several selections on sorted columns). One warp, 33-ary
// search: every step costs one round of 32 independent loads instead of a chain of dependent ones.
__global__ void rq_sorted_tile_range(const unsigned char* col, int width, int64_t tile_stride, int64_t n,
                                     int64_t lo, int64_t hi, uint32_t* out) {
    if (blockIdx.x != 0 || threadIdx.x >= 32) return;
    const int lane = threadIdx.x;
    auto val = [&](int64_t i) -> int64_t {
        const unsigned char* p = col_row(col, width, tile_stride, i);
        if (width == 8) return *reinterpret_cast<const int64_t*>(p);
        if (width == 4) return *reinterpret_cast<const int32_t*>(p);
        return *p;
    };
    // first row whose value is >= key (upper = false) or > key (upper = true)
    auto bound = [&](int64_t key, bool upper, int64_t a, int64_t b) -> int64_t {
        while (a < b) {
            const int64_t step = (b - a + 32) / 33;
            const int64_t p = a + (int64_t)(lane + 1) * step - 1;
            bool left = false;
            if (p < b) { const int64_t v = val(p); left = upper ? (v <= key) : (v < key); }
            const unsigned m = __ballot_sync(kFull, left);
            const int c = __popc(m);               // positions are increasing and `left` is monotone: lanes 0..c-1
            const int64_t na = c > 0 ? a + (int64_t)c * step : a;
            const int64_t pc = a + (int64_t)(c + 1) * step - 1;
            const int64_t nb = (c < 32 && pc < b) ? pc : b;
            a = na; b = nb;
        }
        return a;
    };
    const int64_t r0 = bound(lo, false, 0, n);
    const int64_t r1 = bound(hi, true, r0, n);
    if (lane == 0) {
        const uint32_t t0 = (uint32_t)(r0 / kTile), t1 = (uint32_t)((r1 + kTile - 1) / kTile);
        if (t0 > out[0]) out[0] = t0;
        if (t1 < out[1]) out[1] = t1;
        if (out[1] < out[0]) out[1] = out[0];
    }
}

// shared builds (engine_exec.inl "tile ranges"): population count of the summed bitmap ...
__global__ void rq_popcount_words(const uint32_t* w, size_t n, unsigned long long* out) {
    unsigned long long c = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) c += __popc(w[i]);
    c = (unsigned long long)warp_reduce((int64_t)c, RQ_AGG_SUM);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}
// ... must equal the summed entry count (FlagBlock::entries), else two ranks inserted the same key:
// raise FlagBlock::dup_key so that every rank falls back to the hash form
__global__ void rq_shared_build_check(int32_t* flags) {
    if (threadIdx.x != 0) return;
    const unsigned long long entries = *reinterpret_cast<unsigned long long*>(flags + kFlagWordEntries);
    const unsigned long long bits = *reinterpret_cast<unsigned long long*>(flags + kFlagWordPopcount);
    if (entries != bits) flags[kFlagWordDupKey] = 1;
    if (flags[kFlagWordErr] > 1) flags[kFlagWordErr] = 1;         // (error flags were summed over the ranks)
    if (flags[kFlagWordDupKey] > 1) flags[kFlagWordDupKey] = 1;
}

// min / max of an integer column (upload-time statistics): out[0] = min, out[1] = max
__global__ void rq_col_minmax(const unsigned char* col, int width, int64_t tile_stride, int64_t n, int64_t* out) {
    int64_t lo = INT64_MAX, hi = INT64_MIN;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned char* p = col_row(col, width, tile_stride, i);
        int64_t v;
        if (width == 8) v = *reinterpret_cast<const int64_t*>(p);
        else if (width == 4) v = *reinterpret_cast<const int32_t*>(p);
        else v = *p;
        lo = v < lo ? v : lo;
        hi = v > hi ? v : hi;
    }
    lo = warp_reduce(lo, RQ_AGG_MIN);
    hi = warp_reduce(hi, RQ_AGG_MAX);
    if ((threadIdx.x & 31) == 0) {
        atomicMin((long long*)&out[0], (long long)lo);
        atomicMax((long long*)&out[1], (long long)hi);
    }
}

// re-encodes a chunk of an integer column (plain array, `sw` bytes per value) into its place in a
// tile-major table (`dw` bytes per value): the device side of an upload whose 8-byte columns crossed
// PCIe in a narrower exact encoding (host_narrow.h)
__global__ void rq_repack_col(const unsigned char* src, int sw, unsigned char* dst, int dw, int64_t dstride, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned char* p = src + i * sw;
        int64_t v;
        if (sw == 8) v = *reinterpret_cast<const int64_t*>(p);
        else if (sw == 4) v = *reinterpret_cast<const int32_t*>(p);
        else v = *p;
        unsigned char* q = dst + (i / kTile) * dstride + (i % kTile) * dw;
        if (dw == 8) *reinterpret_cast<int64_t*>(q) = v;
        else if (dw == 4) *reinterpret_cast<int32_t*>(q) = (int32_t)v;
        else *q = (unsigned char)v;
    }
}

// result columns: int64 values -> physical width, strings by value
__global__ void rq_narrow_i32(const int64_t* in, int32_t* out, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int32_t)in[i];
}
__global__ void rq_narrow_i8(const int64_t* in, uint8_t* out, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (uint8_t)in[i];
}
__global__ void rq_gather_str(const int64_t* addrs, unsigned char* out, int width, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const unsigned char* s = reinterpret_cast<const unsigned char*>(addrs[i]);
        unsigned char* d = out + (size_t)i * width;
        int k = 0;
        for (; k < width - 1 && s[k] != 0; k++) d[k] = s[k];
        for (; k < width; k++) d[k] = 0;
    }
}

// Late materialization: fills the deferred output columns of a pipeline from the record its scan
// wrote (engine_exec.inl "late materialization"). Column k reads its reference from record column
// ref[k] and resolves it against one source:
//   LG_ROW    source row r (pair p of a cross source: outer row p / n_inner, inner row p % n_inner)
//             of a fixed-width column: base + (r / 256) * stride + (r % 256) * width, the page layout
//             of owned tables (plain arrays have stride = 256 * width); I32 sign-, I8 zero-extended
//   LG_STR    string column: the address base + r * width, the value the scan's string operand has
//   LG_HASH   hash-table entry i: ent[i * stride + word]
//   LG_DIRECT direct-address entry idx: darr[idx * stride + word], or dlo + idx (word < 0: the payload
//             repeats the key)
// The record's row count is read on the device and clamped to the output's capacity, so replayed and
// graph executions need no host read. One thread per (row, column): the writes of a column coalesce.
enum LateGatherKind : uint8_t { LG_ROW = 0, LG_STR = 1, LG_HASH = 2, LG_DIRECT = 3 };
struct LateCol {
    const unsigned char* base;
    int64_t  stride;        // LG_ROW: bytes per 256-row page; LG_HASH / LG_DIRECT: words per entry
    int64_t  dlo;
    int64_t* out;
    int32_t  word;
    uint8_t  kind, width, ref, side;    // side (cross source): 0 outer, 1 inner, 2 not a cross source
};
struct LateGather {
    LateCol col[kMaxLateOut];
    const int64_t* ref[1 + kMaxProbes];
    const unsigned long long* count;
    int64_t cap;
    const int64_t* cross_inner_rows;    // cross source: row count of the inner relation ...
    int64_t cross_inner_cap;            // ... clamped to its capacity
};
__global__ void rq_late_gather(const __grid_constant__ LateGather G) {
    int64_t n = (int64_t)*G.count;
    if (n > G.cap) n = G.cap;
    const LateCol& c = G.col[blockIdx.y];
    const int64_t* ref = G.ref[c.ref];
    int64_t n_inner = 1;
    if (c.side != 2) {
        n_inner = *G.cross_inner_rows;
        if (n_inner > G.cross_inner_cap) n_inner = G.cross_inner_cap;
        if (n_inner < 1) n_inner = 1;
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t x = ref[i];
        int64_t v;
        if (c.kind == LG_HASH) {
            v = (int64_t)reinterpret_cast<const uint64_t*>(c.base)[(uint64_t)x * (uint64_t)c.stride + c.word];
        } else if (c.kind == LG_DIRECT) {
            v = c.word < 0 ? c.dlo + x : (int64_t)reinterpret_cast<const uint64_t*>(c.base)[(uint64_t)x * (uint64_t)c.stride + c.word];
        } else {
            const uint64_t r = c.side == 2 ? (uint64_t)x : c.side == 1 ? (uint64_t)x % (uint64_t)n_inner : (uint64_t)x / (uint64_t)n_inner;
            if (c.kind == LG_STR) {
                v = (int64_t)(c.base + r * c.width);
            } else {
                const unsigned char* a = c.base + (r / kTile) * (uint64_t)c.stride + (r % kTile) * c.width;
                v = c.width == 8 ? *reinterpret_cast<const int64_t*>(a)
                  : c.width == 4 ? (int64_t)*reinterpret_cast<const int32_t*>(a) : (int64_t)*a;
            }
        }
        c.out[i] = v;
    }
}

// sharded merge: pack the local relation as [ncols][stride] for one all-gather, and unpack the
// gathered [world][ncols][stride] into dense columns in rank order (one launch each instead of
// world x ncols small copies)
struct GatherCols { const int64_t* in[kMaxOut]; int64_t* out[kMaxOut]; int32_t ncols; int32_t world; };
struct GatherCounts { int64_t count[64]; int64_t off[64]; };
__global__ void rq_gather_pack(GatherCols gc, int64_t n, int64_t stride, int64_t* send) {
    const int64_t total = (int64_t)gc.ncols * stride;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t c = i / stride, j = i - c * stride;
        if (j < n) send[i] = gc.in[c][j];
    }
}
__global__ void rq_gather_unpack(GatherCols gc, GatherCounts cnt, int64_t stride, const int64_t* recv) {
    const int64_t per_rank = (int64_t)gc.ncols * stride;
    const int64_t total = per_rank * gc.world;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / per_rank, w = i - r * per_rank;
        const int64_t c = w / stride, j = w - c * stride;
        if (j < cnt.count[r]) gc.out[c][cnt.off[r] + j] = recv[i];
    }
}

// addresses of the rows of a by-value string column (sharded merge: strings arrive by value)
__global__ void rq_str_addrs(const unsigned char* bytes, int width, int64_t n, int64_t* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int64_t)(bytes + (size_t)i * width);
}

// row store (reference DataBlocks, dbdata.h:23-102) -> columns
__global__ void rq_transpose_rows(const unsigned char* rows, int64_t n, int tuple_size, int offset,
                                  int width, unsigned char* col, int64_t tile_stride, int64_t col_row0) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const unsigned char* s = rows + (size_t)i * tuple_size + offset;
        unsigned char* d = const_cast<unsigned char*>(col_row(col, width, tile_stride, col_row0 + i));
        for (int k = 0; k < width; k++) d[k] = s[k];
    }
}

#endif  // __CUDACC_RTC__

}  // namespace rq
