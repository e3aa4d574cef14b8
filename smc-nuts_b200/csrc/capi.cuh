// Shared plumbing of the C-ABI translation units: error string, launch counter, status helpers.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <string>

#include "../../include/smcnuts_b200.h"
#include "common.cuh"
#include "models.cuh"

namespace smcb {

#if defined(SMCB_PLUGIN_TU)
// a generated model plug-in (nuts_plugin.cuh) is its own shared object: it keeps private copies of the small state below
inline std::string& last_error_ref() {
    static thread_local std::string s;
    return s;
}
inline std::atomic<long long> g_launches{0};
#else
std::string& last_error_ref();
extern std::atomic<long long> g_launches;
#endif

inline int fail(const char* where, const char* what) {
    last_error_ref() = std::string(where) + ": " + what;
    return -1;
}
inline int check_launch(const char* where) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(where, cudaGetErrorString(e));
    return 0;
}
#define SMCB_CUDA(call)                                                        \
    do {                                                                       \
        cudaError_t e_ = (call);                                               \
        if (e_ != cudaSuccess) return ::smcb::fail(#call, cudaGetErrorString(e_)); \
    } while (0)
#define SMCB_REQUIRE(cond, msg)                          \
    do {                                                 \
        if (!(cond)) return ::smcb::fail(__func__, msg); \
    } while (0)

// Entry points of a generated model plug-in (nuts_plugin.cuh), resolved by smcb_model_create_plugin; a plug-in built
// against another version of this table is refused
#define SMCB_PLUGIN_ABI 3
struct NutsArgs;
struct PluginVT {
    void* dl;
    int (*abi)(void);
    int (*dim)(void);
    int (*ndata)(void);
    const char* (*last_error)(void);
    long long (*nuts_workspace_bytes)(const ModelDesc*, long long, int);
    int (*nuts_transition)(const ModelDesc*, const NutsArgs*, long long, void*);
    int (*logp_grad)(const ModelDesc*, const double*, long long, double, double*, double*, double*, void*);
    int (*constrained_dim)(void);
    int (*constrain)(const ModelDesc*, const double*, long long, double*, void*);
    int (*gq_dim)(void);
    int (*generated_quantities)(const ModelDesc*, const double*, long long, uint64_t, uint32_t, long long, double*, void*);
};

struct Model {
    ModelDesc desc;
    double* d_data;
    PluginVT* vt = nullptr;   // non-null: a generated model living in its own shared object
    double* d_scale = nullptr; // device copy of the diagonal metric (smcb_model_set_scale)
};

#if defined(SMCB_PLUGIN_TU)
inline int device_sm_count() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}
#else
int device_sm_count();
#endif

// grid for a grid-stride elementwise / reduction kernel: a multiple of the SM count
inline int stride_grid(long long n, int threads, int per_sm) {
    long long want = (n + threads - 1) / threads;
    long long cap = (long long)device_sm_count() * per_sm;
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

}  // namespace smcb
