// K1 + K2 + K3 kernels and their C-ABI: model handles, batched logp/grad, the persistent work-queue NUTS
// transition.  See nuts_lane.cuh for the per-lane algorithm and models.cuh for the densities.
//
// Launch shape: persistent grid = (#SMs x resident CTAs) so every SM keeps its FP64 pipe fed; each lane
// owns one particle at a time and pulls the next index from a global atomic queue (warp-aggregated)
// when its tree ends, which absorbs the 1..2047-leapfrog raggedness of NUTS trees
// (/root/reference/smcnuts/proposal/nuts.py:50-53 loops particles serially instead).
#include <dlfcn.h>

#include <cstdlib>
#include <cstring>
#include <vector>

#include "nuts_builtin.cuh"

namespace smcb {

std::string& last_error_ref() {
    static thread_local std::string s;
    return s;
}
std::atomic<long long> g_launches{0};
static thread_local int g_nuts_blocks_per_sm = 0;   // smcb_nuts_set_blocks_per_sm

int device_sm_count() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

__global__ void combine_logp_kernel(const double* __restrict__ A, const double* __restrict__ B, double phi,
                                    long long N, double* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
        const double lp = A[i] + phi * B[i];
        out[i] = is_finite(lp) ? lp : neg_inf();
    }
}

}  // namespace smcb

using namespace smcb;

extern "C" {

int smcb_version(void) { return 100; }
int smcb_build_flavour(void) { return SMCB_PARITY; }
const char* smcb_last_error(void) { return last_error_ref().c_str(); }
long long smcb_launch_count(void) { return g_launches.load(); }

int smcb_model_create(int kind, const double* host_data, long long n, int dim, void** handle) {
    SMCB_REQUIRE(handle && host_data && n > 0, "null argument");
    std::vector<double> packed;
    ModelDesc d{};
    d.kind = kind;
    if (kind == SMCB_MODEL_ARMA) {
        d.dim = 4; d.T = (int)n;
        packed.assign(host_data, host_data + n);
    } else if (kind == SMCB_MODEL_PRMWCD) {
        SMCB_REQUIRE((n - 1) % 13 == 0, "PRMwCD blob must be [q, y(NO), lgamma(y+1)(NO), X(NO*11)]");
        const int NO = (int)((n - 1) / 13);
        d.dim = 13; d.T = NO; d.q = host_data[0];
        const double *y = host_data + 1, *lg = y + NO, *X = lg + NO;
        packed.assign((size_t)PrmModel::HDR + (size_t)NO * PrmModel::ROW, 0.0);
        for (int i = 0; i < NO; ++i) {
            double* row = packed.data() + PrmModel::HDR + (size_t)i * PrmModel::ROW;
            for (int j = 0; j < 11; ++j) row[j] = X[i * 11 + j];
            row[11] = y[i];
            packed[0] += y[i];
            for (int j = 0; j < 11; ++j) packed[1 + j] += y[i] * X[i * 11 + j];
            packed[12] += lg[i];
        }
        if (PrmModelG<kPrmTiles>::fits(d)) {   // staged block of the tensor-core NUTS kernel, appended to the scalar blob
            const size_t n0 = packed.size();
            packed.resize(n0 + PrmModelG<kPrmTiles>::TOTAL);
            pack_prm_fragments(packed.data(), NO, kPrmTiles, packed.data() + n0);
        }
    } else if (kind == SMCB_MODEL_GAUSS) {
        SMCB_REQUIRE(dim >= 1 && dim <= GaussModel::DMAX && (long long)dim * dim == n, "gauss: need P[D*D], D <= 128");
        d.dim = dim;
        packed.assign(host_data, host_data + n);
        if (dim <= 104) {   // B-fragment packing for the tensor-core NUTS kernel, appended to the plain matrix
            const int nt8 = dim <= 8 ? 1 : dim <= 16 ? 2 : dim <= 32 ? 4 : dim <= 64 ? 8 : 13;
            packed.resize((size_t)n + (size_t)nt8 * 2 * nt8 * 32);
            pack_gauss_fragments(host_data, dim, nt8, packed.data() + n);
        }
    } else {
        return fail("smcb_model_create", "unknown model kind");
    }
    d.n_data = (int)packed.size();
    Model* m = new Model{d, nullptr};
    if (cudaMalloc(&m->d_data, sizeof(double) * packed.size()) != cudaSuccess) {
        delete m;
        return fail("smcb_model_create", "cudaMalloc failed (is a CUDA device present?)");
    }
    SMCB_CUDA(cudaMemcpy(m->d_data, packed.data(), sizeof(double) * packed.size(), cudaMemcpyHostToDevice));
    m->desc.data = m->d_data;
    *handle = m;
    return 0;
}

int smcb_model_create_plugin(const char* so_path, const double* host_data, long long n, void** handle) {
    SMCB_REQUIRE(so_path && handle && n >= 0 && (host_data || n == 0), "null argument");
    void* dl = dlopen(so_path, RTLD_NOW | RTLD_LOCAL);
    if (!dl) return fail("smcb_model_create_plugin", dlerror());
    PluginVT* vt = new PluginVT{};
    vt->dl = dl;
    bool ok = true;
    auto sym = [&](const char* name) { void* p = dlsym(dl, name); ok = ok && p; return p; };
    vt->abi = (int (*)(void))sym("smcb_plugin_abi");
    vt->dim = (int (*)(void))sym("smcb_plugin_dim");
    vt->ndata = (int (*)(void))sym("smcb_plugin_ndata");
    vt->last_error = (const char* (*)(void))sym("smcb_plugin_last_error");
    vt->nuts_workspace_bytes = (long long (*)(const ModelDesc*, long long, int))sym("smcb_plugin_nuts_workspace_bytes");
    vt->nuts_transition = (int (*)(const ModelDesc*, const NutsArgs*, long long, void*))sym("smcb_plugin_nuts_transition");
    vt->logp_grad = (int (*)(const ModelDesc*, const double*, long long, double, double*, double*, double*, void*))sym("smcb_plugin_logp_grad");
    vt->constrained_dim = (int (*)(void))sym("smcb_plugin_constrained_dim");
    vt->constrain = (int (*)(const ModelDesc*, const double*, long long, double*, void*))sym("smcb_plugin_constrain");
    vt->gq_dim = (int (*)(void))sym("smcb_plugin_gq_dim");
    vt->generated_quantities = (int (*)(const ModelDesc*, const double*, long long, uint64_t, uint32_t, long long, double*,
                                        void*))sym("smcb_plugin_generated_quantities");
    auto bail = [&](const char* what) { dlclose(dl); delete vt; return fail("smcb_model_create_plugin", what); };
    if (!ok) return bail("not a model plug-in: an smcb_plugin_* entry point is missing (csrc/nuts_plugin.cuh)");
    if (vt->abi() != SMCB_PLUGIN_ABI) return bail("plug-in ABI version mismatch: rebuild it against this library's csrc/");
    if (vt->ndata() != n) return bail("data blob length differs from the one the plug-in was generated for");
    ModelDesc d{};
    d.kind = kPlugin;
    d.dim = vt->dim();
    d.n_data = (int)n;
    Model* m = new Model{d, nullptr};
    m->vt = vt;
    if (cudaMalloc(&m->d_data, sizeof(double) * (size_t)(n > 0 ? n : 1)) != cudaSuccess) {
        delete m;
        return bail("cudaMalloc failed (is a CUDA device present?)");
    }
    if (n > 0 && cudaMemcpy(m->d_data, host_data, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaFree(m->d_data);
        delete m;
        return bail("cudaMemcpy of the data blob failed");
    }
    m->desc.data = m->d_data;
    *handle = m;
    return 0;
}

int smcb_model_set_scale(void* handle, const double* host_scale) {
    SMCB_REQUIRE(handle, "null argument");
    Model* m = (Model*)handle;
    if (!host_scale) {                       // back to the identity metric
        m->desc.scale = nullptr;
        return 0;
    }
    for (int d = 0; d < m->desc.dim; ++d)
        SMCB_REQUIRE(host_scale[d] > 0.0 && host_scale[d] < 1e300, "scale entries must be positive and finite");
    if (!m->d_scale) SMCB_CUDA(cudaMalloc(&m->d_scale, sizeof(double) * (size_t)m->desc.dim));
    SMCB_CUDA(cudaMemcpy(m->d_scale, host_scale, sizeof(double) * (size_t)m->desc.dim, cudaMemcpyHostToDevice));
    m->desc.scale = m->d_scale;
    return 0;
}

int smcb_model_destroy(void* handle) {
    if (!handle) return 0;
    Model* m = (Model*)handle;
    if (m->d_scale) cudaFree(m->d_scale);
    if (m->vt) {
        dlclose(m->vt->dl);
        delete m->vt;
    }
    cudaFree(m->d_data);
    delete m;
    return 0;
}

int smcb_model_dim(void* handle) { return handle ? ((Model*)handle)->desc.dim : -1; }

int smcb_model_constrained_dim(void* handle) {
    SMCB_REQUIRE(handle && ((Model*)handle)->vt, "bad argument: built-in models constrain inside the moment kernels");
    return ((Model*)handle)->vt->constrained_dim();
}

int smcb_model_constrain(void* handle, const double* x, long long N, double* out, void* stream) {
    SMCB_REQUIRE(handle && ((Model*)handle)->vt, "bad argument: built-in models constrain inside the moment kernels");
    SMCB_REQUIRE(x && out && N >= 0, "bad argument");
    if (N == 0) return 0;
    const Model* m = (const Model*)handle;
    if (m->vt->constrain(&m->desc, x, N, out, stream)) return fail("smcb_model_constrain (plug-in)", m->vt->last_error());
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

int smcb_model_gq_dim(void* handle) {
    SMCB_REQUIRE(handle, "null argument");
    const Model* m = (const Model*)handle;
    return m->vt ? m->vt->gq_dim() : 0;
}

int smcb_model_generated_quantities(void* handle, const double* x, long long N, uint64_t seed, uint32_t counter,
                                    long long particle0, double* out, void* stream) {
    SMCB_REQUIRE(handle && N >= 0 && particle0 >= 0, "bad argument");
    SMCB_REQUIRE(counter < (1u << 24), "bad argument: the call counter has 24 bits");
    const Model* m = (const Model*)handle;
    if (!m->vt || N == 0 || m->vt->gq_dim() == 0) return 0;
    SMCB_REQUIRE(x && out, "bad argument");
    if (m->vt->generated_quantities(&m->desc, x, N, seed, counter, particle0, out, stream))
        return fail("smcb_model_generated_quantities (plug-in)", m->vt->last_error());
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

int smcb_debug_pack_prm(const double* host_scalar_blob, int n_obs, int tiles, double* host_out, long long n_out) {
    SMCB_REQUIRE(host_scalar_blob && host_out && n_obs > 0 && tiles > 0 && n_obs <= 8 * tiles, "bad argument");
    SMCB_REQUIRE(n_out >= 32 + (long long)tiles * 9 * 32, "output too small: 32 + tiles * 288 doubles");
    pack_prm_fragments(host_scalar_blob, n_obs, tiles, host_out);
    return 0;
}

int smcb_logp_grad(void* handle, const double* x, long long N, double phi, double* A, double* B, double* grad,
                   void* stream) {
    SMCB_REQUIRE(handle && x && N >= 0, "bad argument");
    if (N == 0) return 0;
    const Model* m = (const Model*)handle;
    cudaStream_t st = (cudaStream_t)stream;
    if (m->vt) {
        if (m->vt->logp_grad(&m->desc, x, N, phi, A, B, grad, stream)) return fail("smcb_logp_grad (plug-in)", m->vt->last_error());
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return 0;
    }
    switch (m->desc.kind) {
        case kArma: return launch_logp<ArmaModel>(m, x, N, phi, A, B, grad, st);
        case kPRMwCD: return launch_logp<PrmModel>(m, x, N, phi, A, B, grad, st);
        default: return launch_logp<GaussModel>(m, x, N, phi, A, B, grad, st);
    }
}

int smcb_combine_logp(const double* A, const double* B, double phi, long long N, double* out, void* stream) {
    SMCB_REQUIRE(A && B && out && N >= 0, "bad argument");
    if (N == 0) return 0;
    combine_logp_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(A, B, phi, N, out);
    return check_launch("combine_logp_kernel");
}

int smcb_nuts_set_blocks_per_sm(int blocks_per_sm) {
    SMCB_REQUIRE(blocks_per_sm >= 0, "blocks_per_sm must be >= 0 (0 = as many as fit)");
    g_nuts_blocks_per_sm = blocks_per_sm;
    return 0;
}

int smcb_nuts_workspace_bytes(void* handle, long long N, int max_depth, long long* bytes) {
    SMCB_REQUIRE(handle && bytes && N >= 0, "bad argument");
    SMCB_REQUIRE(max_depth >= 1 && max_depth <= 10, "max_depth must be in [1, 10] (reference: MAX_TREE_DEPTH = 10)");
    const Model* m = (const Model*)handle;
    long long b;
    if (m->vt) {
        b = m->vt->nuts_workspace_bytes(&m->desc, N, max_depth);
        if (b < 0) return fail("smcb_nuts_workspace_bytes (plug-in)", "occupancy query failed");
        *bytes = b;
        return 0;
    }
    if (m->desc.scale) {
        b = nuts_ws_bytes_scaled(m, N, max_depth);
        if (b < 0) return fail("smcb_nuts_workspace_bytes", "occupancy query failed");
        *bytes = b;
        return 0;
    }
    switch (m->desc.kind) {
        case kArma: b = nuts_ws_bytes<ArmaModel>(m, N, max_depth); break;
        case kPRMwCD:
            b = prm_use_group(m->desc, N) ? nuts_ws_bytes<PrmModelG<kPrmTiles>>(m, N, max_depth) : nuts_ws_bytes<PrmModel>(m, N, max_depth);
            break;
        default: {
#define WS_G(K) nuts_ws_bytes<GaussModelG<K>>(m, N, max_depth)
            b = SMCB_GAUSS_DISPATCH(m->desc.dim, WS_G, nuts_ws_bytes<GaussModel>(m, N, max_depth));
#undef WS_G
            break;
        }
    }
    if (b < 0) return fail("smcb_nuts_workspace_bytes", "occupancy query failed");
    *bytes = b;
    return 0;
}

int smcb_nuts_transition(void* handle, const double* x, const double* r, long long N, double eps, double phi,
                         int max_depth, int accrej, uint64_t seed, uint32_t iteration, uint64_t particle0,
                         double* x_new, double* r_new, double* A_old, double* B_old, double* A_new, double* B_new,
                         double* ke_old, double* ke_new, int* n_leapfrog, int* accepted, int* depth, double* accept_stat,
                         const double* A_in, const double* B_in, const double* g_in, double* g_new, void* workspace,
                         long long workspace_bytes, void* stream) {
    SMCB_REQUIRE(handle && x && r && x_new && r_new && workspace, "null argument");
    SMCB_REQUIRE((A_in && B_in && g_in) || (!A_in && !B_in && !g_in), "A_in, B_in, g_in: all three or none");
    SMCB_REQUIRE(!(accrej && (g_in || g_new)), "gradient carry-over is not available with the accept-reject epilogue");
    SMCB_REQUIRE(g_new != x_new && (!g_in || (g_in != g_new)), "g_new must not alias its inputs");
    SMCB_REQUIRE(x != x_new && r != r_new, "x_new/r_new must not alias x/r");
    SMCB_REQUIRE(max_depth >= 1 && max_depth <= 10, "max_depth must be in [1, 10] (reference: MAX_TREE_DEPTH = 10)");
    SMCB_REQUIRE(iteration < (1u << 24), "iteration must be < 2^24");
    if (N <= 0) return N == 0 ? 0 : fail("smcb_nuts_transition", "negative N");
    const Model* m = (const Model*)handle;
    NutsArgs a{};
    a.model = m->desc;
    a.x = x; a.r = r; a.N = N; a.eps = eps; a.phi = phi; a.max_depth = max_depth; a.accrej = accrej;
    a.seed = seed; a.iteration = iteration; a.particle0 = particle0;
    a.x_new = x_new; a.r_new = r_new; a.A_old = A_old; a.B_old = B_old; a.A_new = A_new; a.B_new = B_new;
    a.ke_old = ke_old; a.ke_new = ke_new; a.n_leapfrog = n_leapfrog; a.accepted = accepted; a.depth = depth;
    a.accept_stat = accept_stat;
    a.blocks_per_sm = g_nuts_blocks_per_sm;
    a.A_in = A_in; a.B_in = B_in; a.g_in = g_in; a.g_new = g_new;
    a.ws = (double*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    if (m->vt) {
        if (m->vt->nuts_transition(&m->desc, &a, workspace_bytes, stream)) return fail("smcb_nuts_transition (plug-in)", m->vt->last_error());
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return 0;
    }
    if (m->desc.scale) return launch_nuts_scaled(m, a, workspace_bytes, st);
    switch (m->desc.kind) {
        case kArma: return launch_nuts<ArmaModel>(m, a, workspace_bytes, st);
        case kPRMwCD:
            return prm_use_group(m->desc, N) ? launch_nuts<PrmModelG<kPrmTiles>>(m, a, workspace_bytes, st)
                                          : launch_nuts<PrmModel>(m, a, workspace_bytes, st);
        default: {
#define LAUNCH_G(K) launch_nuts<GaussModelG<K>>(m, a, workspace_bytes, st)
            return SMCB_GAUSS_DISPATCH(m->desc.dim, LAUNCH_G, launch_nuts<GaussModel>(m, a, workspace_bytes, st));
#undef LAUNCH_G
        }
    }
}

}  // extern "C"
