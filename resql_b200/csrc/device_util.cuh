// Device helpers shared by the kernels: mbarrier / TMA PTX, string semantics, hashing.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/resql_b200.h"
#include "rq_internal.h"

namespace rq {

// ------------------------------------------------------------------------------------------
// device memory: stream-ordered allocations from the default pool (release threshold raised at
// rq_init), so that per-query hash tables and intermediates are recycled instead of going
// through cudaMalloc / cudaFree every time
// ------------------------------------------------------------------------------------------
#ifndef __CUDACC_RTC__     // (host code: not part of a run-time compiled specialization, jit.h)
inline cudaStream_t& alloc_stream() { static cudaStream_t s = nullptr; return s; }
template <typename T>
inline cudaError_t dmalloc(T** p, size_t bytes) {
    return cudaMallocAsync(reinterpret_cast<void**>(p), bytes ? bytes : 1, alloc_stream());
}
inline void dfree(void* p) {
    if (p) cudaFreeAsync(p, alloc_stream());
}
#endif

// ------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + TMA bulk copy
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// (all on 32-bit shared-space addresses)
__device__ __forceinline__ void mbar_init_s(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx_s(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s_s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
        : "memory");
}
// L2 eviction policy for data that is streamed exactly once (scanned columns): evict first, so
// that hash tables and Bloom filters stay resident in the 126 MB L2 under a multi-GB scan
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void tma_bulk_g2s_hint(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar,
                                                  uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(policy)
        : "memory");
}
// bring a global range into L2 ahead of the bulk copy that will stage it (no shared memory needed)
__device__ __forceinline__ void tma_prefetch_l2(const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
// one lane of the (converged) warp; ptxas then issues a following bulk copy once instead of
// looping over the active lanes
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void mbar_wait_s(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "RQ_WAIT_S:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra RQ_DONE_S;\n"
        "bra RQ_WAIT_S;\n"
        "RQ_DONE_S:\n"
        "}" ::"r"(bar),
        "r"(parity)
        : "memory");
}

// ------------------------------------------------------------------------------------------
// string semantics (qlib/scalar.h)
// ------------------------------------------------------------------------------------------
// compareChar (qlib/scalar.h:27-46): equal after ignoring trailing blanks on either side
__device__ __forceinline__ int64_t str_eq_char(const char* a, const char* b) {
    while (*a != '\0' && *b != '\0') {
        if (*a != *b) return 0;
        a++; b++;
    }
    while (*a != '\0') { if (*a != ' ') return 0; a++; }
    while (*b != '\0') { if (*b != ' ') return 0; b++; }
    return 1;
}
// compareVarchar (qlib/scalar.h:16-24): exact
__device__ __forceinline__ int64_t str_eq_varchar(const char* a, const char* b) {
    while (*a != '\0' && *b != '\0') {
        if (*a != *b) return 0;
        a++; b++;
    }
    return (*a == *b) ? 1 : 0;
}
// stringLikeCheck(string, like) (qlib/scalar.h:57-120), restated statement by statement in index
// form. The reference matches the literal prefix and the literal suffix of the pattern
// independently (they may overlap: 'aba' like 'ab%ba' is true), then scans the infix pieces left
// to right; '_' matches any one character (cmpLike :50-54). Behaviour that follows from its code is
// kept ('%%' accepts nothing, '%_' accepts everything, '' like '%a' is true); pinned against the
// reference engine by tests/golden/like_matrix.json.
__device__ __forceinline__ bool like_cmp(char c, char l) { return c == l || l == '_'; }
__device__ __noinline__ int64_t str_like(const char* s, const char* p) {
    int s_end = 0, p_end = 0;
    while (s[s_end] != '\0') s_end++;
    while (p[p_end] != '\0') p_end++;
    int l_in_start = 0, l_in_end = p_end, s_in_start = 0, s_in_end = s_end;
    int l_pos = 0, s_pos = 0;
    if (p[0] != '%') {                                  // prefix
        for (; l_pos < p_end && s_pos < s_end && p[l_pos] != '%'; ++l_pos, ++s_pos)
            if (!like_cmp(s[s_pos], p[l_pos])) return 0;
        l_in_start = l_pos;
        s_in_start = s_pos;
    }
    if (l_in_start == p_end) return s_in_start == s_end ? 1 : 0;     // no-'%' likes
    if (p[p_end - 1] != '%') {                          // suffix
        s_pos = s_end - 1;
        l_pos = p_end - 1;
        for (; l_pos >= 0 && s_pos >= 0 && p[l_pos] != '%'; --l_pos, --s_pos)
            if (!like_cmp(s[s_pos], p[l_pos])) return 0;
        l_in_end = l_pos;
        s_in_end = s_pos + 1;
    }
    if (l_in_start < l_in_end) {                        // infixes
        l_pos = l_in_start + 1;
        s_pos = s_in_start;
        while (s_pos < s_in_end && l_pos < l_in_end) {
            int l_trace = l_pos, s_trace = s_pos;
            while (like_cmp(s[s_trace], p[l_trace]) && s_trace < s_in_end) {
                ++l_trace;
                if (p[l_trace] == '%') {
                    l_pos = ++l_trace;
                    s_pos = s_trace;
                    break;
                }
                ++s_trace;
            }
            ++s_pos;
        }
    }
    return l_pos >= l_in_end ? 1 : 0;
}

__device__ __forceinline__ uint64_t mix64(uint64_t h) {
    h ^= h >> 33; h *= 0xff51afd7ed558ccdULL;
    h ^= h >> 33; h *= 0xc4ceb9fe1a85ec53ULL;
    h ^= h >> 33;
    return h;
}

__device__ __forceinline__ int64_t agg_identity(int kind) {
    if (kind == RQ_AGG_MIN) return INT64_MAX;
    if (kind == RQ_AGG_MAX) return INT64_MIN;
    return 0;
}

// signed truncating division like x86 idiv; b == 0 raises the runtime error flag
__device__ __forceinline__ int64_t div_trunc(int64_t a, int64_t b, int32_t* err) {
    if (b == 0) { *err = 1; return 0; }
    if (b == -1) return (int64_t)(0ULL - (uint64_t)a);   // avoids INT64_MIN / -1 trap semantics
    return a / b;
}


}  // namespace rq
