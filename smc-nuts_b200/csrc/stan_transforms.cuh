// Stan's constraining transforms of the vector parameter types (Stan Reference Manual, "Constraint transforms"), their
// log-Jacobians and the pullbacks of their gradients.  The model structs that smcnuts/model/stan_codegen.py generates call
// these for `simplex[K]`, `ordered[K]` and `positive_ordered[K]` parameters, from eval() (density) and constrain()
// (estimates), so nvcc (plug-in) and g++ (host tests) compile the same arithmetic.
//
// Conventions: y -> the unconstrained coordinates of one vector (K - 1 for a simplex, K otherwise), x -> its K constrained
// values.  *_constrain writes x and returns log |J| (ok turns false when a value under- or overflows: the density is then
// -inf).  *_pullback maps gx = d f / d x to gy = d f / d y + d log|J| / d y, in O(K).
//
// simplex is the stick-breaking transform of Stan releases up to 2.35 (and of BridgeStan builds against them):
//   z_k = inv_logit(y_k - log(K - k)),  x_k = r_k z_k,  r_1 = 1,  r_{k+1} = r_k (1 - z_k),  x_K = r_K,
//   log J = sum_{k<K} [log z_k + log(1 - z_k) + log r_k] = sum_{k<K} [log z_k + (K - k) log(1 - z_k)].
// r is carried as a product of the 1 - z_k, each formed as inv_logit(-u), and log z / log(1 - z) as -log1p_exp(-u) /
// -log1p_exp(u): at |y| ~ 30 the values, log J and the gradient stay accurate (1 - sum x would cancel there).
#pragma once
#include <cmath>

#include "common.cuh"

namespace smcb {
namespace stan {

// z = inv_logit(u) and 1 - z = inv_logit(-u), each in the two-branch form, from one exp: e = exp(-|u|), d = 1 + e
struct Logistic {
    double e, z, zc;
    SMCB_HD explicit Logistic(double u) : e(exp(-fabs(u))) {
        const double d = 1.0 + e;
        z = u >= 0.0 ? 1.0 / d : e / d;
        zc = u >= 0.0 ? e / d : 1.0 / d;
    }
};

// ---- ordered (x_1 = y_1) and positive_ordered (x_1 = exp(y_1)):  x_k = x_{k-1} + exp(y_k)
template <int K, bool POSITIVE>
SMCB_HD double ordered_constrain(const double* y, double* x, bool& ok) {
    double lj = 0.0;
    if (POSITIVE) {
        const double e = exp(y[0]);
        x[0] = e;
        lj += y[0];
        ok = ok && e > 0.0 && e < INFINITY;
    } else {
        x[0] = y[0];
    }
#pragma unroll
    for (int k = 1; k < K; ++k) {
        const double e = exp(y[k]);
        x[k] = x[k - 1] + e;
        lj += y[k];
        ok = ok && e > 0.0 && x[k] < INFINITY;
    }
    return lj;
}

// gy_k = exp(y_k) sum_{j>=k} gx_j  (+ 1 from log J for every coordinate that enters through exp)
template <int K, bool POSITIVE>
SMCB_HD void ordered_pullback(const double* y, const double* gx, double* gy) {
    double s = 0.0;
#pragma unroll
    for (int k = K - 1; k >= 1; --k) {
        s += gx[k];
        gy[k] = s * exp(y[k]) + 1.0;
    }
    s += gx[0];
    gy[0] = POSITIVE ? s * exp(y[0]) + 1.0 : s;
}

// ---- simplex (stick-breaking)
template <int K>
SMCB_HD double simplex_constrain(const double* y, double* x, bool& ok) {
    double lj = 0.0, r = 1.0, log_r = 0.0;
#pragma unroll
    for (int k = 0; k < K - 1; ++k) {
        const double u = y[k] - log((double)(K - 1 - k));
        const Logistic s(u);
        const double l = log1p(s.e);                                 // log z = -log1p_exp(-u), log(1 - z) = -log1p_exp(u)
        const double log_z = -((u < 0.0 ? -u : 0.0) + l), log_1mz = -((u > 0.0 ? u : 0.0) + l);
        x[k] = r * s.z;
        lj += log_z + log_1mz + log_r;
        r *= s.zc;
        log_r += log_1mz;
    }
    x[K - 1] = r;
    ok = ok && lj > -INFINITY && lj < INFINITY;
    return lj;
}

// reverse sweep with the adjoint a of the remaining stick r_{k+1}:
//   gy_k = x_k (1 - z_k) (gx_k - a) + (1 - z_k) - (K - k) z_k,   a <- gx_k z_k + a (1 - z_k)
template <int K>
SMCB_HD void simplex_pullback(const double* y, const double* x, const double* gx, double* gy) {
    double a = gx[K - 1];
#pragma unroll
    for (int k = K - 2; k >= 0; --k) {
        const Logistic s(y[k] - log((double)(K - 1 - k)));
        gy[k] = x[k] * s.zc * (gx[k] - a) + s.zc - (double)(K - 1 - k) * s.z;
        a = gx[k] * s.z + a * s.zc;
    }
}

}  // namespace stan
}  // namespace smcb
