// TEST TOOL ONLY: runs the 4-lanes-per-particle NUTS kernels (PrmModelG / GaussModelG + the group paths of
// csrc/nuts_lane.cuh) on the CPU through the fiber-based warp emulator of simt_emu.h, so the `not gpu` test-suite can
// check the tensor-core fragment dataflow, the group folds and the warp-level work queue against the oracle.
// The loop below restates nuts_transition_kernel (csrc/nuts_kernel.cu) for ONE persistent warp.
// Never loaded by the product package; the product path has no CPU fallback.
#define SMCB_SIMT_EMU 1
#include "simt_emu.h"

#include "../../smc-nuts_b200/csrc/nuts_lane.cuh"

using namespace smcb;

template <class M>
static void run_warp_kernel(NutsArgs a, const double* staged);

// the diagonal-metric wrapper of the same kernel when the caller passed a scale
template <class M>
static void run_maybe_scaled(NutsArgs a, const double* staged) {
    if (a.model.scale) run_warp_kernel<ScaledModel<M>>(a, staged);
    else run_warp_kernel<M>(a, staged);
}

template <class M>
static void run_warp_kernel(NutsArgs a, const double* staged) {
    constexpr int G = M::GROUP;
    const int rec = nuts_ws_doubles(M(a.model, staged).nloc(), a.max_depth, a.g_new != nullptr);
    std::vector<double> ws((size_t)simt_emu::kLanes * rec, 0.0);
    const int stride = nuts_stage_stride(M(a.model, staged).nloc());
    std::vector<double> stage((size_t)simt_emu::kLanes * stride, 0.0);   // the staging rows of the device kernel's shared memory
    unsigned long long head = 0;
    simt_emu::run_warp([&](int lane_id) {
        M model(a.model, staged);
        Lane<M> lane;
        lane.idle_init(model, lane_id % G);
        lane.stg = stage.data() + (size_t)lane_id * stride;
        double* w = ws.data() + (size_t)lane_id * rec;
        constexpr unsigned kLeaders = G == 1 ? 0xffffffffu : 0x11111111u;
        const unsigned group_first = (unsigned)lane_id & ~(unsigned)(G - 1);
        bool drained = false;
        for (;;) {
            const bool want = (lane.phase == kIdle) && !drained;
            const unsigned m = __ballot_sync(0xffffffffu, want) & kLeaders;
            if (m) {
                const int leader = __builtin_ffs((int)m) - 1;
                unsigned long long base = 0;
                if (lane_id == leader) {
                    base = head;
                    head += (unsigned long long)__builtin_popcount(m);
                }
                base = __shfl_sync(0xffffffffu, base, leader);
                if (want) {
                    const long long p = (long long)base + __builtin_popcount(m & ((1u << group_first) - 1u));
                    if (p < a.N) lane.begin(a, model, p, w);
                    else drained = true;
                }
            }
            if (__all_sync(0xffffffffu, lane.phase == kIdle)) break;
            if (lane.phase != kIdle) { lane.pre_eval(a); lane.prefetch_ck(); }
            double A, B, g[M::NLOC];
            model.eval(lane.xa, a.phi, A, B, g);
            lane.take_grad(g);
            if (lane.phase != kIdle) lane.post_eval(a, A, B);
        }
    });
}

// kind 1: PRMwCD (data = scalar blob [16 header][T rows of 12]); kind 2: Gaussian (data = P, dim x dim)
extern "C" int hostsim_nuts_simt(int kind, const double* data, int n_data, int dim, int T, double q, const double* x,
                                 const double* r, long long N, double eps, double phi, int max_depth, int accrej,
                                 unsigned long long seed, unsigned iteration, unsigned long long particle0,
                                 double* x_new, double* r_new, double* A_old, double* B_old, double* A_new, double* B_new,
                                 double* ke_old, double* ke_new, int* n_leapfrog, int* accepted, int* depth,
                                 const double* scale) {
    NutsArgs a;
    std::memset(&a, 0, sizeof a);
    a.model = ModelDesc{kind, dim, n_data, T, q, data, scale};
    a.x = x; a.r = r; a.N = N; a.eps = eps; a.phi = phi; a.max_depth = max_depth; a.accrej = accrej;
    a.seed = seed; a.iteration = iteration; a.particle0 = particle0;
    a.x_new = x_new; a.r_new = r_new; a.A_old = A_old; a.B_old = B_old; a.A_new = A_new; a.B_new = B_new;
    a.ke_old = ke_old; a.ke_new = ke_new; a.n_leapfrog = n_leapfrog; a.accepted = accepted; a.depth = depth;
    if (kind == kPRMwCD) {
        using M = PrmModelG<13>;
        if (!M::fits(a.model)) return -1;
        std::vector<double> staged(M::TOTAL);
        pack_prm_fragments(data, T, 13, staged.data());
        run_maybe_scaled<M>(a, staged.data());
        return 0;
    }
    if (kind == kGauss) {
        const int nt8 = dim <= 8 ? 1 : dim <= 16 ? 2 : dim <= 32 ? 4 : dim <= 64 ? 8 : 13;
        if (dim > 104) return -1;
        std::vector<double> staged((size_t)nt8 * 2 * nt8 * 32);
        pack_gauss_fragments(data, dim, nt8, staged.data());
        switch (nt8) {
            case 1: run_maybe_scaled<GaussModelG<1>>(a, staged.data()); break;
            case 2: run_maybe_scaled<GaussModelG<2>>(a, staged.data()); break;
            case 4: run_maybe_scaled<GaussModelG<4>>(a, staged.data()); break;
            case 8: run_maybe_scaled<GaussModelG<8>>(a, staged.data()); break;
            default: run_maybe_scaled<GaussModelG<13>>(a, staged.data()); break;
        }
        return 0;
    }
    return -1;
}

// A probe model for the diagonal-metric wrapper alone: it hands back the x it is evaluated at as its gradient (A = B = 0),
// so ScaledModel<Probe>::eval returns g = s * (s * z) slot by slot, padded slots included -- the per-lane coordinate map
// (slot i of lane `sub` is coordinate sub + GROUP * i) and the scale 1 of the padding, with no NUTS tree in between.
template <int G, int NL>
struct ProbeModel {
    static constexpr int DMAX = G * NL, STATIC_D = 0, GROUP = G, NLOC = NL, STATIC_NL = NL;
    static constexpr bool STAGE = false;
    int D;
    explicit ProbeModel(const ModelDesc& d, const double*) : D(d.dim) {}
    int dim() const { return D; }
    constexpr int nloc() const { return NL; }
    void eval(const double (&x)[NL], double, double& A, double& B, double (&g)[NL]) const {
        for (int i = 0; i < NL; ++i) g[i] = x[i];
        A = B = 0.0;
    }
};

template <int G, int NL>
static void probe(int dim, const double* scale, const double* z, double* g) {
    ModelDesc d{};
    d.dim = dim;
    d.scale = scale;
    simt_emu::run_warp([&](int lane) {
        ScaledModel<ProbeModel<G, NL>> m(d, nullptr);
        double zl[NL], gl[NL], A, B;
        for (int i = 0; i < NL; ++i) zl[i] = z[lane * NL + i];
        m.eval(zl, 1.0, A, B, gl);
        for (int i = 0; i < NL; ++i) g[lane * NL + i] = gl[i];
    });
}

// z, g: [32 lanes][nloc] slot values.  group 4 with nloc = 4 (PrmModelG) or 2 NT8 (GaussModelG<NT8>); group 1 with nloc 4.
extern "C" int hostsim_scaled_probe(int group, int nloc, int dim, const double* scale, const double* z, double* g) {
    if (group == 1 && nloc == 4) probe<1, 4>(dim, scale, z, g);
    else if (group == 4 && nloc == 2) probe<4, 2>(dim, scale, z, g);
    else if (group == 4 && nloc == 4) probe<4, 4>(dim, scale, z, g);
    else if (group == 4 && nloc == 8) probe<4, 8>(dim, scale, z, g);
    else if (group == 4 && nloc == 16) probe<4, 16>(dim, scale, z, g);
    else if (group == 4 && nloc == 26) probe<4, 26>(dim, scale, z, g);
    else return -1;
    return 0;
}
