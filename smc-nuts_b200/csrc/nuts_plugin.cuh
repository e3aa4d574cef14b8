// Model plug-in: one generated (or hand-written) model struct compiled into its own shared object together with the
// NUTS / logp kernel templates of nuts_launch.cuh.  The product library loads it with smcb_model_create_plugin and routes
// smcb_logp_grad, smcb_nuts_workspace_bytes and smcb_nuts_transition of that model handle through the entry points below;
// every model-agnostic kernel (weights, resampling, L-kernels, estimators) is the library's own.  smcb_model_constrain
// routes through smcb_plugin_constrain: the struct's constrain() over rows of particles; smcb_model_generated_quantities
// through smcb_plugin_generated_quantities: the generated-quantities struct over rows of particles.
//
// Replaces the generic half of /root/reference/smcnuts/model/bridgestan.py:13-26 (any Stan program through BridgeStan):
// smcnuts/model/stan_codegen.py writes the struct, smcnuts/model/generated.py writes and compiles a translation unit
//
//     #define SMCB_PLUGIN_TU 1
//     #include "nuts_plugin.cuh"
//     #include "model_gen.cuh"          // struct GenModel { ... eval(x, phi, A, B, g) ... }
//     #include "model_gq.cuh"           // struct GenModelGQ { ... generated_quantities(x, rng, out) ... }
//     SMCB_DEFINE_PLUGIN(GenModel)
//     SMCB_DEFINE_PLUGIN_GQ(GenModelGQ)
//
// with nvcc -gencode arch=compute_100a,code=sm_100a.
#pragma once
#ifndef SMCB_PLUGIN_TU
#error "define SMCB_PLUGIN_TU before including nuts_plugin.cuh"
#endif
#include "nuts_launch.cuh"
#include "stan_rng.cuh"

namespace smcb {

// Constrained rows of a plug-in model: one thread per particle, CONSTRAIN_NT particles per block.  The block's x rows and
// its out rows are staged through shared memory (row stride padded to an odd number of doubles: no bank conflicts when each
// thread walks its own row), so that both the loads and the stores of global memory are coalesced.
constexpr int CONSTRAIN_NT = 64;

template <class M>
__global__ void __launch_bounds__(CONSTRAIN_NT) plugin_constrain_kernel(const double* __restrict__ x, long long N,
                                                                        double* __restrict__ out) {
    constexpr int D = M::DMAX, C = M::CDIM, S = (D > C ? D : C) | 1;
    extern __shared__ double rows[];                                 // [CONSTRAIN_NT][S]
    const long long row0 = (long long)blockIdx.x * CONSTRAIN_NT;
    const int nrows = (int)(N - row0 < CONSTRAIN_NT ? N - row0 : CONSTRAIN_NT);
    for (int e = threadIdx.x; e < nrows * D; e += CONSTRAIN_NT) rows[(e / D) * S + e % D] = x[row0 * D + e];
    __syncthreads();
    double xr[D], cr[C];
    const int t = threadIdx.x;
    if (t < nrows) {
#pragma unroll
        for (int d = 0; d < D; ++d) xr[d] = rows[t * S + d];
    }
    __syncthreads();
    if (t < nrows) {
        M::constrain(xr, cr);
#pragma unroll
        for (int c = 0; c < C; ++c) rows[t * S + c] = cr[c];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < nrows * C; e += CONSTRAIN_NT) out[row0 * C + e] = rows[(e / C) * S + e % C];
}

template <class M>
int launch_constrain(const double* x, long long N, double* out, cudaStream_t st) {
    constexpr int S = (M::DMAX > M::CDIM ? M::DMAX : M::CDIM) | 1;
    const size_t smem = sizeof(double) * CONSTRAIN_NT * S;
    if (smem > 48 * 1024)
        SMCB_CUDA(cudaFuncSetAttribute(plugin_constrain_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long blocks = (N + CONSTRAIN_NT - 1) / CONSTRAIN_NT;
    plugin_constrain_kernel<M><<<(unsigned)blocks, CONSTRAIN_NT, smem, st>>>(x, N, out);
    return check_launch("plugin_constrain_kernel");
}

// Generated quantities of a plug-in model, laid out like plugin_constrain_kernel: one thread per particle, the x rows and
// the out rows of a block staged through shared memory (odd row stride) so that global loads and stores coalesce.  Rows
// wider than the shared-memory budget allows for 64 particles are staged for fewer particles per block (ROWS < 64: the
// other threads of the block idle); stan_codegen.py caps G so that one row always fits.  Row i draws from the stream of
// particle particle0 + i.
template <class Q>
struct GqLayout {
    static constexpr int S = (Q::DMAX > Q::GDIM ? Q::DMAX : Q::GDIM) | 1;
    static constexpr int BUDGET = 200 * 1024 / 8;                    // doubles of dynamic shared memory per block
    static_assert(S <= BUDGET, "a generated-quantities row must fit in shared memory");
    static constexpr int ROWS = BUDGET / S < CONSTRAIN_NT ? BUDGET / S : CONSTRAIN_NT;
    static constexpr size_t SMEM = sizeof(double) * ROWS * S;
};

template <class Q>
__global__ void __launch_bounds__(CONSTRAIN_NT) plugin_gq_kernel(Q q, const double* __restrict__ x, long long N,
                                                                 uint64_t seed, uint32_t counter, long long particle0,
                                                                 double* __restrict__ out) {
    using L = GqLayout<Q>;
    constexpr int D = Q::DMAX, G = Q::GDIM, S = L::S;
    extern __shared__ double rows[];                                 // [ROWS][S]
    const long long row0 = (long long)blockIdx.x * L::ROWS;
    const int nrows = (int)(N - row0 < L::ROWS ? N - row0 : L::ROWS);
    const int t = threadIdx.x;
    double xr[D];
    for (int e = t; e < nrows * D; e += CONSTRAIN_NT) rows[(e / D) * S + e % D] = x[row0 * D + e];
    __syncthreads();
    if (t < nrows) {
#pragma unroll
        for (int d = 0; d < D; ++d) xr[d] = rows[t * S + d];
    }
    __syncthreads();
    if (t < nrows) {
        stan::Rng rng(seed, counter, (uint64_t)(particle0 + row0 + t));
        q.generated_quantities(xr, rng, &rows[t * S]);
    }
    __syncthreads();
    constexpr int GW = G > 0 ? G : 1;                                // (no rows to write when G = 0)
    for (int e = t; e < nrows * G; e += CONSTRAIN_NT) out[row0 * G + e] = rows[(e / GW) * S + e % GW];
}

template <class Q>
int launch_gq(const ModelDesc& d, const double* x, long long N, uint64_t seed, uint32_t counter, long long particle0,
              double* out, cudaStream_t st) {
    using L = GqLayout<Q>;
    if (Q::GDIM == 0 || N == 0) return 0;
    if (L::SMEM > 48 * 1024)
        SMCB_CUDA(cudaFuncSetAttribute(plugin_gq_kernel<Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::SMEM));
    const long long blocks = (N + L::ROWS - 1) / L::ROWS;
    plugin_gq_kernel<Q><<<(unsigned)blocks, CONSTRAIN_NT, L::SMEM, st>>>(Q(d), x, N, seed, counter, particle0, out);
    return check_launch("plugin_gq_kernel");
}

}  // namespace smcb

// launch shape of a plug-in model: 128 threads, two CTAs per SM (its register need is unknown; wide models spill)
#define SMCB_DEFINE_PLUGIN(MODEL)                                                                                        \
    namespace smcb {                                                                                                     \
    template <> struct LaunchCfg<MODEL> { static constexpr int NT = 128, MIN_BLOCKS = 2; };                              \
    }                                                                                                                    \
    extern "C" {                                                                                                         \
    int smcb_plugin_abi(void) { return SMCB_PLUGIN_ABI; }                                                                \
    int smcb_plugin_dim(void) { return MODEL::STATIC_D; }                                                                \
    int smcb_plugin_ndata(void) { return MODEL::NDATA; }                                                                 \
    const char* smcb_plugin_last_error(void) { return smcb::last_error_ref().c_str(); }                                  \
    long long smcb_plugin_nuts_workspace_bytes(const smcb::ModelDesc* d, long long N, int max_depth) {                   \
        smcb::Model m{*d, nullptr};                                                                                      \
        if (d->scale) return smcb::nuts_ws_bytes<smcb::ScaledModel<MODEL>>(&m, N, max_depth);                            \
        return smcb::nuts_ws_bytes<MODEL>(&m, N, max_depth);                                                             \
    }                                                                                                                    \
    int smcb_plugin_nuts_transition(const smcb::ModelDesc* d, const smcb::NutsArgs* a, long long ws_bytes, void* st) {   \
        smcb::Model m{*d, nullptr};                                                                                      \
        if (d->scale) return smcb::launch_nuts<smcb::ScaledModel<MODEL>>(&m, *a, ws_bytes, (cudaStream_t)st);            \
        return smcb::launch_nuts<MODEL>(&m, *a, ws_bytes, (cudaStream_t)st);                                             \
    }                                                                                                                    \
    int smcb_plugin_logp_grad(const smcb::ModelDesc* d, const double* x, long long N, double phi, double* A, double* B,  \
                              double* g, void* st) {                                                                     \
        smcb::Model m{*d, nullptr};                                                                                      \
        return smcb::launch_logp<MODEL>(&m, x, N, phi, A, B, g, (cudaStream_t)st);                                       \
    }                                                                                                                    \
    int smcb_plugin_constrained_dim(void) { return MODEL::CDIM; }                                                        \
    int smcb_plugin_constrain(const smcb::ModelDesc*, const double* x, long long N, double* out, void* st) {             \
        return smcb::launch_constrain<MODEL>(x, N, out, (cudaStream_t)st);                                               \
    }                                                                                                                    \
    }

// the generated quantities of a plug-in model: a struct with DMAX, GDIM, a constructor from the ModelDesc and
// generated_quantities(x, rng, out) (stan_codegen.py writes `<model struct>GQ`; GDIM = 0 when the program has none)
#define SMCB_DEFINE_PLUGIN_GQ(GQ)                                                                                        \
    extern "C" {                                                                                                         \
    int smcb_plugin_gq_dim(void) { return GQ::GDIM; }                                                                    \
    int smcb_plugin_generated_quantities(const smcb::ModelDesc* d, const double* x, long long N, uint64_t seed,          \
                                         uint32_t counter, long long particle0, double* out, void* st) {                \
        return smcb::launch_gq<GQ>(*d, x, N, seed, counter, particle0, out, (cudaStream_t)st);                           \
    }                                                                                                                    \
    }
