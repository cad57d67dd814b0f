// Run-time specialization of the scan kernel.
//
// Everything the interpreter in rq_scan_kernel decides per tile from KParams - the program, the
// operand kinds and offsets, the sink and its aggregate forms, the stage layout, the probe flags - is
// known on the host when a pipeline is launched. Here the same scan_kernel.cuh source the library was
// built from (embedded at build time, jit_sources.inc) is compiled once per pipeline with NVRTC, with
// those fields as compile-time constants (a FixedSpec, generated from the RQ_SPEC_FIELDS list): the
// unit loop unrolls, every unit's switch folds to its one case and the sink keeps only its form.
//
// A specialization is cached under its generated source, which spells out every baked field: a launch
// whose fields differ gets another specialization, so results are those of the generic kernel by
// construction. The register-aggregation and generic variants (<4>, <1>, <0>) are specialized; the
// cross, late and round variants, a missing libnvrtc and a failed compile keep the ahead-of-time
// kernels (the last two say so once on stderr).
#pragma once
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include "rq_internal.h"
#include "scan_kernel.cuh"

namespace rq {

// the kernel's headers as the library was built from them: kJitHeaderName[i] (the name an #include
// uses) and kJitHeaderText[i]
#include "jit_sources.inc"

// what NVRTC lacks of the C and CUDA headers the kernel's headers include
static const char kJitStdint[] =
    "#pragma once\n"
    "typedef signed char int8_t; typedef short int16_t; typedef int int32_t; typedef long long int64_t;\n"
    "typedef unsigned char uint8_t; typedef unsigned short uint16_t; typedef unsigned int uint32_t;\n"
    "typedef unsigned long long uint64_t; typedef unsigned long long uintptr_t;\n"
    "#define INT64_MAX 0x7fffffffffffffffLL\n#define INT64_MIN (-INT64_MAX - 1)\n";
static const char kJitEmpty[] = "#pragma once\n";     // (NVRTC defines size_t itself)

typedef int (*nvrtc_create_t)(void**, const char*, const char*, int, const char* const*, const char* const*);
typedef int (*nvrtc_compile_t)(void*, int, const char* const*);
typedef int (*nvrtc_size_t)(void*, size_t*);
typedef int (*nvrtc_get_t)(void*, char*);
typedef int (*nvrtc_destroy_t)(void**);
typedef const char* (*nvrtc_error_t)(int);

struct Nvrtc {
    bool tried = false;
    void* lib = nullptr;
    nvrtc_create_t create = nullptr;
    nvrtc_compile_t compile = nullptr;
    nvrtc_size_t log_size = nullptr, cubin_size = nullptr;
    nvrtc_get_t log = nullptr, cubin = nullptr;
    nvrtc_destroy_t destroy = nullptr;
    nvrtc_error_t error = nullptr;
};

struct JitKernel {
    cudaLibrary_t lib = nullptr;
    cudaKernel_t kernel = nullptr;    // null: the specialization failed, the generic kernel runs
};

struct Jit {
    std::mutex mu;                            // the cache and NVRTC
    Nvrtc nv;
    std::map<std::string, JitKernel> cache;   // spec_key -> loaded specialization
    bool warned = false, warned_many = false;
    std::atomic<unsigned long long> launches{0};   // launches that ran a specialization
    std::atomic<unsigned long long> captured{0};   // ... of them recorded into a stream capture (graph)
    double compile_ms = 0;                    // NVRTC time of all specializations so far
};
// More specializations than this in one process means some baked field varies from launch to launch
// (a data-dependent layout or flag); each new one costs a compile, so it is reported once.
static constexpr size_t kJitManySpecs = 64;
static Jit g_jit;

// libnvrtc is opened at run time (like libnccl, dist.h), so the library has no link dependency on it
static bool nvrtc_load(Nvrtc& n, std::string& err) {
    if (n.tried) { if (!n.lib) err = "libnvrtc.so.12 not found"; return n.lib != nullptr; }
    n.tried = true;
    const char* names[] = {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12"};
    for (const char* nm : names)
        if ((n.lib = dlopen(nm, RTLD_NOW | RTLD_LOCAL)) != nullptr) break;
    if (!n.lib) { err = "libnvrtc.so.12 not found"; return false; }
    n.create = (nvrtc_create_t)dlsym(n.lib, "nvrtcCreateProgram");
    n.compile = (nvrtc_compile_t)dlsym(n.lib, "nvrtcCompileProgram");
    n.log_size = (nvrtc_size_t)dlsym(n.lib, "nvrtcGetProgramLogSize");
    n.log = (nvrtc_get_t)dlsym(n.lib, "nvrtcGetProgramLog");
    n.cubin_size = (nvrtc_size_t)dlsym(n.lib, "nvrtcGetCUBINSize");
    n.cubin = (nvrtc_get_t)dlsym(n.lib, "nvrtcGetCUBIN");
    n.destroy = (nvrtc_destroy_t)dlsym(n.lib, "nvrtcDestroyProgram");
    n.error = (nvrtc_error_t)dlsym(n.lib, "nvrtcGetErrorString");
    if (!n.create || !n.compile || !n.log_size || !n.log || !n.cubin_size || !n.cubin || !n.destroy || !n.error) {
        dlclose(n.lib);
        n.lib = nullptr;
        err = "libnvrtc lacks required symbols";
        return false;
    }
    return true;
}

// ---- the fixed spec ----------------------------------------------------------------------------------
static std::string spec_lit(int v) { return std::to_string(v); }
static std::string spec_lit(uint32_t v) { return std::to_string(v) + "u"; }
static std::string spec_lit(bool v) { return v ? "true" : "false"; }
static std::string spec_lit(VRef v) {
    return "VRef{" + std::to_string(v.kind) + ", " + std::to_string(v.slot) + ", " + std::to_string(v.off16) + "}";
}
static bool spec_zero(int v) { return v == 0; }
static bool spec_zero(uint32_t v) { return v == 0; }
static bool spec_zero(bool v) { return !v; }
static bool spec_zero(VRef v) { return v.kind == 0 && v.slot == 0 && v.off16 == 0; }

// The cache key of a launch: the bytes of every baked field (the program without its immediates, then
// the RQ_SPEC_FIELDS values) and the variant. Cheaper than generating the source on every launch.
template <typename T>
static void spec_put(std::string& k, T v) { k.append(reinterpret_cast<const char*>(&v), sizeof v); }
static std::string spec_key(const KParams& P, int gr) {
    std::string k;
    k.reserve(1024);
    spec_put(k, gr);
    spec_put(k, P.n_insn);
    for (int i = 0; i < P.n_insn; i++) {
        UInsn u = P.insn[i];
        u.imm = 0;
        spec_put(k, u);
    }
#define RQ_KEY_FIELD(T, NAME, EXPR) spec_put(k, (T)(EXPR));
#define RQ_KEY_ARRAY(T, NAME, N, EXPR) for (int i = 0; i < (N); i++) spec_put(k, (T)(EXPR));
#define RQ_KEY_PROBE(T, NAME, EXPR) for (int p = 0; p < kMaxProbes; p++) { const DProbe& pr = P.probe[p]; spec_put(k, (T)(EXPR)); }
#define RQ_KEY_PROBE2(T, NAME, N, EXPR) \
    for (int p = 0; p < kMaxProbes; p++) { const DProbe& pr = P.probe[p]; for (int i = 0; i < (N); i++) spec_put(k, (T)(EXPR)); }
    RQ_SPEC_FIELDS(RQ_KEY_FIELD, RQ_KEY_ARRAY, RQ_KEY_PROBE, RQ_KEY_PROBE2)
#undef RQ_KEY_FIELD
#undef RQ_KEY_ARRAY
#undef RQ_KEY_PROBE
#undef RQ_KEY_PROBE2
    return k;
}

// The mangled name of rq_scan_kernel<gr> (the non-cross, non-late, non-round variants)
static std::string spec_kernel_name(int gr) {
    return "_ZN2rq14rq_scan_kernelILi" + std::to_string(gr) + "ELb0ELb0ELb0EEEvNS_7KParamsE";
}

// The source of one specialization: FixedSpec with the baked fields of P, selected as RQ_SCAN_SPEC, and
// the explicit instantiation of rq_scan_kernel<gr> over it (the same kernel as the library's, with its
// fields as constants). Immediates stay in KParams (FixedSpec::insn reads them from the launch's
// parameters, where they are constant-bank operands).
static std::string spec_source(const KParams& P, int gr) {
    std::string s = "#include \"rq_internal.h\"\nnamespace rq {\nstruct FixedSpec {\n    static constexpr bool kFixed = true;\n";
    s += "    static __device__ __forceinline__ UInsn insn(const KParams& P, uint32_t, int pc) {\n        UInsn u{};\n        switch (pc) {\n";
    for (int i = 0; i < P.n_insn; i++) {
        const UInsn& u = P.insn[i];
        char line[256];
        snprintf(line, sizeof line, "        case %d: u = UInsn{%d, %d, %d, %d, %d, %d, %d, 0, %uu, %uu, 0, %uu, %uu}; break;\n", i, u.code,
                 u.flags, u.gop, u.aux, u.xkind, u.ykind, u.zkind, u.xrel, u.dstrel, u.yrel, u.zrel);
        s += line;
    }
    s += "        }\n        u.imm = P.insn[pc].imm;\n        return u;\n    }\n";
    const std::string fn = "    static __device__ __forceinline__ constexpr ";
#define RQ_GEN_FIELD(T, NAME, EXPR) s += fn + #T " " #NAME "(const KParams&) { return " + spec_lit((T)(EXPR)) + "; }\n";
#define RQ_GEN_ARRAY(T, NAME, N, EXPR)                                                              \
    {                                                                                               \
        s += fn + #T " " #NAME "(const KParams&, int i) { switch (i) {";                          \
        for (int i = 0; i < (N); i++)                                                               \
            if (!spec_zero((T)(EXPR))) s += " case " + std::to_string(i) + ": return " + spec_lit((T)(EXPR)) + ";"; \
        s += " default: return " #T "{}; } }\n";                                                    \
    }
#define RQ_GEN_PROBE(T, NAME, EXPR)                                                                 \
    {                                                                                               \
        s += fn + #T " " #NAME "(const DProbe&, int p) { switch (p) {";                           \
        for (int p = 0; p < kMaxProbes; p++) {                                                      \
            const DProbe& pr = P.probe[p];                                                          \
            if (!spec_zero((T)(EXPR))) s += " case " + std::to_string(p) + ": return " + spec_lit((T)(EXPR)) + ";"; \
        }                                                                                           \
        s += " default: return " #T "{}; } }\n";                                                    \
    }
#define RQ_GEN_PROBE2(T, NAME, N, EXPR)                                                             \
    {                                                                                               \
        s += fn + #T " " #NAME "(const DProbe&, int p, int i) { switch (p * 256 + i) {";          \
        for (int p = 0; p < kMaxProbes; p++) {                                                      \
            const DProbe& pr = P.probe[p];                                                          \
            for (int i = 0; i < (N); i++)                                                           \
                if (!spec_zero((T)(EXPR))) s += " case " + std::to_string(p * 256 + i) + ": return " + spec_lit((T)(EXPR)) + ";"; \
        }                                                                                           \
        s += " default: return " #T "{}; } }\n";                                                    \
    }
    RQ_SPEC_FIELDS(RQ_GEN_FIELD, RQ_GEN_ARRAY, RQ_GEN_PROBE, RQ_GEN_PROBE2)
#undef RQ_GEN_FIELD
#undef RQ_GEN_ARRAY
#undef RQ_GEN_PROBE
#undef RQ_GEN_PROBE2
    s += "};\n}  // namespace rq\n#define RQ_SCAN_SPEC FixedSpec\n#include \"scan_kernel.cuh\"\n";
    s += "template __global__ void rq::rq_scan_kernel<" + std::to_string(gr) + ">(const __grid_constant__ rq::KParams);\n";
    return s;
}

// Compiles a specialization for sm_100a. verbose: ptxas reports registers, stack and spills in the log.
static bool spec_compile(const std::string& src, bool verbose, std::string& cubin, std::string& log) {
    Nvrtc& n = g_jit.nv;
    if (!nvrtc_load(n, log)) return false;
    std::vector<const char*> names, texts;
    for (size_t i = 0; i < sizeof(kJitHeaderName) / sizeof(kJitHeaderName[0]); i++) {
        names.push_back(kJitHeaderName[i]);
        texts.push_back(kJitHeaderText[i]);
    }
    names.push_back("stdint.h"); texts.push_back(kJitStdint);
    names.push_back("stddef.h"); texts.push_back(kJitEmpty);
    names.push_back("cuda_runtime.h"); texts.push_back(kJitEmpty);
    void* prog = nullptr;
    int rc = n.create(&prog, src.c_str(), "rq_scan_spec.cu", (int)names.size(), texts.data(), names.data());
    if (rc != 0) { log = std::string("nvrtcCreateProgram: ") + n.error(rc); return false; }
    // the Makefile's device options: sm_100a, -O3 (NVRTC's default), C++17; the C ABI's prototypes
    // in resql_b200.h are declared, not called, so they may default to device functions
    std::vector<const char*> opts = {"-arch=sm_100a", "-std=c++17", "-lineinfo", "-default-device"};
    if (verbose) opts.push_back("-Xptxas=-v");
    rc = n.compile(prog, (int)opts.size(), opts.data());
    size_t ls = 0;
    n.log_size(prog, &ls);
    log.assign(ls, '\0');
    if (ls) n.log(prog, &log[0]);
    while (!log.empty() && log.back() == '\0') log.pop_back();
    if (rc == 0) {
        size_t cs = 0;
        n.cubin_size(prog, &cs);
        cubin.assign(cs, '\0');
        n.cubin(prog, &cubin[0]);
    } else {
        log = std::string("nvrtcCompileProgram: ") + n.error(rc) + "\n" + log;
    }
    n.destroy(&prog);
    return rc == 0;
}

// The specialization of a launch of variant gr with parameters P, compiled and loaded on first use
// (null: run the generic kernel). Launches inside a stream capture only use what is cached.
static cudaKernel_t spec_kernel(const KParams& P, int gr, bool capturing, int smem_max) {
    const std::string key = spec_key(P, gr);
    std::lock_guard<std::mutex> lk(g_jit.mu);
    auto it = g_jit.cache.find(key);
    if (it != g_jit.cache.end()) return it->second.kernel;
    if (capturing) return nullptr;
    if (g_jit.cache.size() >= kJitManySpecs && !g_jit.warned_many) {
        fprintf(stderr, "resql_b200: %zu scan kernel specializations compiled in this process\n", g_jit.cache.size());
        g_jit.warned_many = true;
    }
    JitKernel jk;
    std::string cubin, log;
    const auto t0 = std::chrono::steady_clock::now();
    const bool ok = spec_compile(spec_source(P, gr), false, cubin, log);
    g_jit.compile_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (ok && cudaLibraryLoadData(&jk.lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0) == cudaSuccess &&
        cudaLibraryGetKernel(&jk.kernel, jk.lib, spec_kernel_name(gr).c_str()) == cudaSuccess &&
        cudaFuncSetAttribute((const void*)jk.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max) == cudaSuccess) {
        g_jit.cache[key] = jk;
        return jk.kernel;
    }
    if (ok) log = std::string("loading the specialization: ") + cudaGetErrorString(cudaGetLastError());
    if (jk.lib) cudaLibraryUnload(jk.lib);
    if (!g_jit.warned) {
        fprintf(stderr, "resql_b200: scan kernel specialization unavailable, the generic kernels run (%s)\n",
                log.substr(0, log.find('\n')).c_str());
        g_jit.warned = true;
    }
    g_jit.cache[key] = JitKernel();
    return nullptr;
}

}  // namespace rq
