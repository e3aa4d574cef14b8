// TEST TOOL ONLY: compiles the device lane state machine (smc-nuts_b200/csrc/nuts_lane.cuh) with g++ and
// runs `lanes` simulated lanes against a shared work queue on the CPU, so the `not gpu` test-suite can
// check the kernel LOGIC (tree bookkeeping, draw order, refill) against the oracle without a GPU.
// Never loaded by the product package; the product path has no CPU fallback.
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../smc-nuts_b200/csrc/nuts_lane.cuh"

using namespace smcb;

template <class M>
static void run(NutsArgs a, int lanes) {
    const int rec = nuts_ws_doubles(M(a.model, a.model.data).nloc(), a.max_depth, a.g_new != nullptr);
    std::vector<double> ws((size_t)lanes * rec, 0.0);
    std::vector<Lane<M>> L(lanes);
    M model(a.model, a.model.data);
    for (auto& l : L) { l.idle_init(model, 0); l.stg = nullptr; }
    long long head = 0;
    for (;;) {
        bool any = false;
        for (int i = 0; i < lanes; ++i) {
            Lane<M>& l = L[i];
            if (l.phase == kIdle && head < a.N) l.begin(a, model, head++, ws.data() + (size_t)i * rec);
            if (l.phase == kIdle) continue;
            any = true;
            l.pre_eval(a);
            l.prefetch_ck();
            double A, B, g[M::NLOC];
            model.eval(l.xa, a.phi, A, B, g);
            l.take_grad(g);
            l.post_eval(a, A, B);
        }
        if (!any) break;
    }
}

extern "C" int hostsim_nuts(int kind, const double* data, int n_data, int dim, int T, double q, const double* x,
                            const double* r, long long N, double eps, double phi, int max_depth, int accrej,
                            unsigned long long seed, unsigned iteration, unsigned long long particle0, double* x_new,
                            double* r_new, double* A_old, double* B_old, double* A_new, double* B_new, double* ke_old,
                            double* ke_new, int* n_leapfrog, int* accepted, int* depth, const double* A_in,
                            const double* B_in, const double* g_in, double* g_new, int lanes, const double* scale) {
    NutsArgs a;
    std::memset(&a, 0, sizeof a);
    a.model = ModelDesc{kind, dim, n_data, T, q, data, scale};
    a.x = x; a.r = r; a.N = N; a.eps = eps; a.phi = phi; a.max_depth = max_depth; a.accrej = accrej;
    a.seed = seed; a.iteration = iteration; a.particle0 = particle0;
    a.x_new = x_new; a.r_new = r_new; a.A_old = A_old; a.B_old = B_old; a.A_new = A_new; a.B_new = B_new;
    a.ke_old = ke_old; a.ke_new = ke_new; a.n_leapfrog = n_leapfrog; a.accepted = accepted; a.depth = depth;
    a.A_in = A_in; a.B_in = B_in; a.g_in = g_in; a.g_new = g_new;
    if (scale) {   // diagonal metric: x, x_new are z = x / scale (the caller converts, as proposal/nuts.py does)
        if (kind == kArma) run<ScaledModel<ArmaModel>>(a, lanes);
        else if (kind == kPRMwCD) run<ScaledModel<PrmModel>>(a, lanes);
        else run<ScaledModel<GaussModel>>(a, lanes);
    } else {
        if (kind == kArma) run<ArmaModel>(a, lanes);
        else if (kind == kPRMwCD) run<PrmModel>(a, lanes);
        else run<GaussModel>(a, lanes);
    }
    return 0;
}
