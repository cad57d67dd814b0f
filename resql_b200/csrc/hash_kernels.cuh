// Hash tables in HBM: join build/probe and high-cardinality GROUP BY.
// Replaces src/qlib/hash.h of the reference (linear probing with a stored hash per entry,
// :385-478) and its users hashjoin.h:118-279 / aggregation.h:240-295. Entries are packed rows
// [tag][key words][payload / accumulator words] padded to a multiple of 32 bytes; tag 0 = empty,
// 1 = being written, else hash|2.
#pragma once
#include <cuda_runtime.h>
#include "rq_internal.h"
#include "device_util.cuh"

namespace rq {

struct HashTableDev {
    DHashTable d{};
    uint64_t capacity = 0;
    uint64_t entries = 0;       // occupied slots after the build
    ~HashTableDev() {
        dfree(d.ent); dfree(d.bloom); dfree(d.dbits); dfree(d.darr);
    }
};

constexpr uint64_t kTagLocked = 1ULL;
// A full table is detected by its LOAD (entries are counted per warp tile against DHashTable::limit,
// scan_kernel.cuh), not by the length of a probe run: a join key with thousands of duplicates makes
// long runs in a nearly empty table (hashjoin.h:226-256 keeps every duplicate). Walks only give up
// when somebody raised the table-full flag.
constexpr uint64_t kFullCheckEvery = 256;
// A claim that had to walk this far (duplicates, or keys clustering under the order-preserving hash)
// raises FlagBlock::dup_key; `full` points at FlagBlock::ht_full (rq_internal.h)
constexpr uint64_t kLongRun = 1024;
__device__ __forceinline__ void note_long_run(const int32_t* full) { *const_cast<int32_t*>(full + kDupKeyFromHtFull) = 1; }

// key kinds: 0 integer word, 1 CHAR (equality ignores trailing blanks), 2 VARCHAR (exact)
__device__ __forceinline__ uint64_t hash_str(const unsigned char* s, bool strip) {
    // FNV-1a over the bytes; for CHAR the trailing blanks are left out so that values equal
    // under compareChar hash alike
    int len = 0, last = 0;
    while (s[len] != 0) { if (s[len] != ' ') last = len + 1; len++; }
    const int n = strip ? last : len;
    uint64_t h = 0xcbf29ce484222325ULL;
    for (int i = 0; i < n; i++) { h ^= s[i]; h *= 0x100000001b3ULL; }
    return h;
}

__device__ __forceinline__ uint64_t hash_typed(const int64_t* k, const uint8_t* kind, int nk) {
    uint64_t h = 0x9E3779B97F4A7C15ULL;
    for (int j = 0; j < nk; j++) {
        uint64_t w = (kind[j] == 0) ? (uint64_t)k[j]
                                    : hash_str(reinterpret_cast<const unsigned char*>(k[j]), kind[j] == 1);
        h = mix64(h ^ w) + 0x9E3779B97F4A7C15ULL;
    }
    return h;
}

// Hash of a key tuple. One integer key (the usual join / group key) takes a single 64-bit
// multiply, (key - hsub) * hmul: Fibonacci hashing or the order-preserving scaling of a dense key
// domain (see DHashTable); the home slot comes from the HIGH bits. Composite and string keys go
// through the mixing hash.
__device__ __forceinline__ uint64_t hash_int(const DHashTable& ht, int64_t k) {
    return ((uint64_t)k - (uint64_t)ht.hsub) * ht.hmul;
}
__device__ __forceinline__ uint64_t hash_keys(const DHashTable& ht, const int64_t* k) {
    if (ht.nk == 1 && ht.key_kind[0] == 0) return hash_int(ht, k[0]);
    return hash_typed(k, ht.key_kind, ht.nk);
}
// blocked Bloom filter: word index and the two bits inside the 32-bit block
__device__ __forceinline__ uint32_t bloom_word(const DHashTable& ht, uint64_t h) {
    const uint64_t g = h ^ (h >> 29);
    return (uint32_t)(g >> 10) & ht.bloom_mask;
}
__device__ __forceinline__ uint32_t bloom_bits(const DHashTable& ht, uint64_t h) {
    (void)ht;
    const uint64_t g = h ^ (h >> 29);
    return (1u << ((uint32_t)g & 31)) | (1u << ((uint32_t)(g >> 5) & 31));
}

__device__ __forceinline__ bool key_word_equal(int64_t a, int64_t b, int kind) {
    if (kind == 0) return a == b;
    if (kind == 1) return str_eq_char(reinterpret_cast<const char*>(a), reinterpret_cast<const char*>(b)) != 0;
    return str_eq_varchar(reinterpret_cast<const char*>(a), reinterpret_cast<const char*>(b)) != 0;
}

__device__ __forceinline__ uint64_t* ht_entry(const DHashTable& ht, uint64_t i) {
    return ht.ent + i * ht.stride;
}

__device__ __forceinline__ bool slot_keys_equal(const DHashTable& ht, uint64_t i, const int64_t* k) {
    const volatile uint64_t* e = ht_entry(ht, i);
    for (int j = 0; j < ht.nk; j++)
        if (!key_word_equal((int64_t)e[1 + j], k[j], ht.key_kind[j])) return false;
    return true;
}

// join build: every tuple gets its own slot (duplicates are kept, hashjoin.h:226-256)
__device__ __forceinline__ bool ht_insert_dup(const DHashTable& ht, const int64_t* k, uint64_t h,
                                              uint64_t* slot_out, const int32_t* full) {
    const uint64_t tag = h | 2ULL;
    const uint64_t cap = ht.cap_mask + 1;
    uint64_t i = h >> ht.shift;
    for (uint64_t tries = 0; tries < cap; tries++) {
        uint64_t* e = ht_entry(ht, i);
        const unsigned long long old = atomicCAS((unsigned long long*)e, 0ULL, (unsigned long long)tag);
        if (old == 0ULL) {
            for (int j = 0; j < ht.nk; j++) e[1 + j] = (uint64_t)k[j];
            *slot_out = i;
            return true;
        }
        i = (i + 1) & ht.cap_mask;
        if ((tries & (kFullCheckEvery - 1)) == kFullCheckEvery - 1 && *(volatile int32_t*)full) return false;
    }
    return false;
}

// the same, starting the walk at slot `i` (the home slot was already found taken); keys are
// written by the caller
__device__ __forceinline__ bool ht_insert_dup_from(const DHashTable& ht, uint64_t h, uint64_t i,
                                                   uint64_t* slot_out, const int32_t* full) {
    const uint64_t tag = h | 2ULL;
    const uint64_t cap = ht.cap_mask + 1;
    for (uint64_t tries = 1; tries < cap; tries++) {
        const unsigned long long old = atomicCAS((unsigned long long*)ht_entry(ht, i), 0ULL, (unsigned long long)tag);
        if (old == 0ULL) { *slot_out = i; return true; }
        i = (i + 1) & ht.cap_mask;
        if (tries == kLongRun) note_long_run(full);
        if ((tries & (kFullCheckEvery - 1)) == kFullCheckEvery - 1 && *(volatile int32_t*)full) return false;
    }
    return false;
}

// GROUP BY: find the slot of the key or claim a new one (aggregation.h:262-279)
__device__ __forceinline__ bool ht_find_or_insert(const DHashTable& ht, const int64_t* k, uint64_t h,
                                                  uint64_t* slot_out, bool* fresh, const int32_t* full) {
    const uint64_t tag = h | 2ULL;
    const uint64_t cap = ht.cap_mask + 1;
    uint64_t i = h >> ht.shift;
    for (uint64_t tries = 0; tries < cap; tries++) {
        if ((tries & (kFullCheckEvery - 1)) == kFullCheckEvery - 1 && *(volatile int32_t*)full) return false;
        volatile uint64_t* e = ht_entry(ht, i);
        uint64_t t = e[0];
        if (t == 0ULL) {
            t = atomicCAS((unsigned long long*)e, 0ULL, (unsigned long long)kTagLocked);
            if (t == 0ULL) {
                for (int j = 0; j < ht.nk; j++) e[1 + j] = (uint64_t)k[j];
                __threadfence();
                atomicExch((unsigned long long*)e, (unsigned long long)tag);
                *slot_out = i;
                *fresh = true;
                return true;
            }
        }
        while (t == kTagLocked) t = e[0];
        if (t == tag) {
            __threadfence();
            if (slot_keys_equal(ht, i, k)) { *slot_out = i; return true; }
        }
        i = (i + 1) & ht.cap_mask;
    }
    return false;
}

// ---- helper kernels ------------------------------------------------------------------------
// clear the tags and set the accumulators of a hash-aggregation table to their identities
struct HtKinds { uint8_t kind[kMaxAggs]; };
__global__ void rq_ht_init(DHashTable ht, HtKinds kinds, int init_vals) {
    const uint64_t cap = ht.cap_mask + 1;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cap) {
        uint64_t* e = ht_entry(ht, i);
        e[0] = 0;
        const int first = ht.packed ? 1 : 1 + ht.nk;
        if (init_vals)
            for (int a = 0; a < ht.nv; a++) e[first + a] = (uint64_t)agg_identity(kinds.kind[a]);
    }
}

// occupied slots -> dense int64 columns. colmap[c] < nk selects key word colmap[c], otherwise
// accumulator colmap[c]-nk (duplicate aggregates share one accumulator).
struct HtCompact { int32_t colmap[kMaxOut]; int64_t* out[kMaxOut]; };
__global__ void rq_ht_compact(DHashTable ht, HtCompact hc, int n_out,
                              unsigned long long* count, unsigned long long out_cap) {
    const uint64_t cap = ht.cap_mask + 1;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool used = i < cap && *ht_entry(ht, i) != 0ULL;
    const unsigned bal = __ballot_sync(0xffffffffu, used);
    if (!bal) return;
    const int lane = threadIdx.x & 31;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(count, (unsigned long long)__popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (used) {
        const unsigned long long pos = base + __popc(bal & ((1u << lane) - 1));
        const uint64_t* e = ht_entry(ht, i);
        if (pos < out_cap)       // (sized from a count the host may only have predicted)
            for (int c = 0; c < n_out; c++) hc.out[c][pos] = (int64_t)e[1 + hc.colmap[c]];
    }
}

// the same for tables whose entries carry the packed group key in their first word
struct PackedCompact {
    int32_t nk;                     // logical key columns
    uint8_t shift[kMaxKeys], bits[kMaxKeys], sign[kMaxKeys];
    int32_t n_out;
    int32_t colmap[kMaxOut];        // < nk: key column, else accumulator colmap - nk
    int64_t* out[kMaxOut];
};
__global__ void rq_ht_compact_packed(DHashTable ht, PackedCompact pc, unsigned long long* count, unsigned long long out_cap) {
    const uint64_t cap = ht.cap_mask + 1;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool used = i < cap && *ht_entry(ht, i) != 0ULL;
    const unsigned bal = __ballot_sync(0xffffffffu, used);
    if (!bal) return;
    const int lane = threadIdx.x & 31;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(count, (unsigned long long)__popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (used) {
        const unsigned long long pos = base + __popc(bal & ((1u << lane) - 1));
        if (pos >= out_cap) return;
        const uint64_t* e = ht_entry(ht, i);
        const uint64_t k = e[0] - 1;
        for (int c = 0; c < pc.n_out; c++) {
            const int m = pc.colmap[c];
            if (m < pc.nk) {
                const int b = pc.bits[m];
                uint64_t f = (b >= 64) ? k : ((k >> pc.shift[m]) & ((1ULL << b) - 1));
                if (pc.sign[m] && b < 64 && ((f >> (b - 1)) & 1)) f |= ~((1ULL << b) - 1);
                pc.out[c][pos] = (int64_t)f;
            } else {
                pc.out[c][pos] = (int64_t)e[1 + (m - pc.nk)];
            }
        }
    }
}

// groupjoin (IMPL_GROUPJOIN): the touched entries of a direct-address table -> dense int64 columns.
// word[c] < 0 selects the entry's key (dlo + index), otherwise entry word word[c] (a stored payload or
// an accumulator). A block of kGjThreads threads covers kGjWordsPerThread words per thread of the
// touched bitmap and takes its output range with ONE atomic: the groups are sparse in the bitmap (Q3
// at SF100: 1.1 M groups in 18.75 M words), so one atomic per warp would be ~0.5 M atomics on one
// counter, which serialize.
constexpr int kGjThreads = 256, kGjWordsPerThread = 8;
struct GjCompact { int32_t n_out; int16_t word[kMaxOut]; int64_t* out[kMaxOut]; };
__global__ void __launch_bounds__(kGjThreads) rq_groupjoin_compact(DHashTable ht, const uint32_t* touched, GjCompact gc,
                                                                   unsigned long long* count, unsigned long long out_cap) {
    __shared__ int warp_off[kGjThreads / 32];
    __shared__ unsigned long long block_base;
    const uint64_t words = (ht.dsize + 31) / 32;
    const uint64_t w0 = (uint64_t)blockIdx.x * kGjThreads * kGjWordsPerThread + threadIdx.x;
    uint32_t w[kGjWordsPerThread];
    int n = 0;
#pragma unroll
    for (int j = 0; j < kGjWordsPerThread; j++) {
        const uint64_t i = w0 + (uint64_t)j * kGjThreads;
        w[j] = i < words ? touched[i] : 0u;
        n += __popc(w[j]);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_off[warp] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int k = 0; k < kGjThreads / 32; k++) { const int x = warp_off[k]; warp_off[k] = t; t += x; }
        block_base = t ? atomicAdd(count, (unsigned long long)t) : 0ULL;
    }
    __syncthreads();
    unsigned long long pos = block_base + (unsigned long long)(warp_off[warp] + incl - n);
#pragma unroll 1
    for (int j = 0; j < kGjWordsPerThread; j++) {
        const uint64_t i = w0 + (uint64_t)j * kGjThreads;
        for (uint32_t b = w[j]; b; b &= b - 1, pos++) {
            const uint64_t idx = i * 32 + (uint64_t)(__ffs(b) - 1);
            if (pos >= out_cap) continue;          // (sized from a count the host may only have predicted)
            const uint64_t* e = ht.darr + idx * ht.dnv;
            for (int c = 0; c < gc.n_out; c++)
                gc.out[c][pos] = gc.word[c] < 0 ? ht.dlo + (int64_t)idx : (int64_t)e[gc.word[c]];
        }
    }
}

}  // namespace rq
