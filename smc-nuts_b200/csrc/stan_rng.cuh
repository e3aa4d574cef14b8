// Stan's `_rng` functions for the `generated quantities` block of generated models (Stan Functions Reference).  The gq
// structs that smcnuts/model/stan_codegen.py generates call these per element, so nvcc (plug-in) and g++ (host tests)
// compile the same arithmetic.
//
// Randomness: one Philox stream per particle, stream id kStreamGQ, keyed by (seed, call counter, GLOBAL particle index):
// a particle's draws do not depend on N, the shard, the row order or the launch shape.  Draws are read in order from
// that stream (StreamReader); rejection loops simply read further.
//
// Invalid arguments (where Stan's _rng throws: a non-positive scale, a probability outside [0, 1], a Poisson rate at or
// above 2^30, ...) return NaN and clear Rng::ok; the generated code then writes NaN to every output of the particle.
// Every loop is bounded: a rejection loop that has not accepted after kMaxTrials trials fails the same way.
//
// Algorithms: inversion where a closed form exists; normal by Box-Muller as in stream_normal_pair; gamma by
// Marsaglia-Tsang (2000) with the u^(1/alpha) boost for alpha < 1, beta from two gammas; Poisson by inversion below a
// mean of 10 and PTRS (Hoermann 1993) above; binomial by inversion below n min(p, 1 - p) = 10 and BTRS (Hoermann 1993)
// above; neg_binomial_2 as Poisson(Gamma).
#pragma once
#include <cmath>
#include <cstdint>

#include "philox.cuh"

namespace smcb {
namespace stan {

constexpr int kMaxTrials = 1000;
constexpr double kPoissonMaxRate = 1073741824.0;     // 2^30, Stan's POISSON_MAX_RATE

struct Rng {
    uint64_t seed, particle;
    uint32_t iter_stream;
    StreamReader r;
    bool ok;
    SMCB_HD Rng(uint64_t seed_, uint32_t counter, uint64_t particle_)
        : seed(seed_), particle(particle_), iter_stream((counter << 8) | kStreamGQ), ok(true) {
        r.reset();
    }
    // u in [0, 1), numpy's double construction (as the library's other streams)
    SMCB_HD double unit() { return (double)r.next_bits(seed, iter_stream, particle) * 0x1.0p-53; }
    // u in (0, 1): for logarithms and divisions
    SMCB_HD double open() { return ((double)(r.next_bits(seed, iter_stream, particle) >> 1) + 0.5) * 0x1.0p-52; }
    SMCB_HD double fail() {
        ok = false;
        return NAN;
    }
};

SMCB_HD bool finite(double v) { return fabs(v) < INFINITY; }
SMCB_HD bool positive(double v) { return v > 0.0 && v < INFINITY; }

// ---- continuous
SMCB_HD double std_normal_rng(Rng& g) {
    const double u1 = g.unit(), u2 = g.unit();
    return sqrt(-2.0 * log1p(-u1)) * cos(kTwoPi * u2);
}

SMCB_HD double normal_rng(double mu, double sigma, Rng& g) {
    if (!(finite(mu) && positive(sigma))) return g.fail();
    return mu + sigma * std_normal_rng(g);
}

SMCB_HD double lognormal_rng(double mu, double sigma, Rng& g) {
    if (!(finite(mu) && positive(sigma))) return g.fail();
    return exp(mu + sigma * std_normal_rng(g));
}

SMCB_HD double cauchy_rng(double mu, double sigma, Rng& g) {
    if (!(finite(mu) && positive(sigma))) return g.fail();
    return mu + sigma * tan(0.5 * kTwoPi * (g.open() - 0.5));
}

SMCB_HD double double_exponential_rng(double mu, double sigma, Rng& g) {
    if (!(finite(mu) && positive(sigma))) return g.fail();
    const double w = g.open() - 0.5;
    return mu - sigma * copysign(1.0, w) * log1p(-2.0 * fabs(w));
}

SMCB_HD double logistic_rng(double mu, double sigma, Rng& g) {
    if (!(finite(mu) && positive(sigma))) return g.fail();
    const double u = g.open();
    return mu + sigma * (log(u) - log1p(-u));
}

SMCB_HD double exponential_rng(double beta, Rng& g) {
    if (!positive(beta)) return g.fail();
    return -log(g.open()) / beta;
}

SMCB_HD double uniform_rng(double a, double b, Rng& g) {
    if (!(finite(a) && finite(b) && a < b)) return g.fail();
    return a + (b - a) * g.unit();
}

// Gamma(a, 1) for a >= 1: Marsaglia & Tsang, "A simple method for generating gamma variables" (2000)
SMCB_HD double gamma_mt(double a, Rng& g) {
    const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    for (int it = 0; it < kMaxTrials; ++it) {
        const double z = std_normal_rng(g);
        double v = 1.0 + c * z;
        if (v <= 0.0) continue;
        v = v * v * v;
        const double u = g.open(), z2 = z * z;
        if (u < 1.0 - 0.0331 * z2 * z2 || log(u) < 0.5 * z2 + d * (1.0 - v + log(v))) return d * v;
    }
    return g.fail();
}

// Gamma(a, 1) for a > 0 and its logarithm (a < 1: Gamma(a + 1) u^(1/a); the logarithm stays finite where the value
// underflows)
SMCB_HD double gamma_unit(double a, Rng& g) {
    if (a >= 1.0) return gamma_mt(a, g);
    const double x = gamma_mt(a + 1.0, g);
    return x * pow(g.open(), 1.0 / a);
}

SMCB_HD double log_gamma_unit(double a, Rng& g) {
    if (a >= 1.0) return log(gamma_mt(a, g));
    const double x = gamma_mt(a + 1.0, g);
    return log(x) + log(g.open()) / a;
}

SMCB_HD double gamma_rng(double alpha, double beta, Rng& g) {
    if (!(positive(alpha) && positive(beta))) return g.fail();
    return gamma_unit(alpha, g) / beta;
}

SMCB_HD double inv_gamma_rng(double alpha, double beta, Rng& g) {
    if (!(positive(alpha) && positive(beta))) return g.fail();
    return beta / gamma_unit(alpha, g);
}

SMCB_HD double beta_rng(double a, double b, Rng& g) {
    if (!(positive(a) && positive(b))) return g.fail();
    if (a >= 1.0 && b >= 1.0) {
        const double x = gamma_mt(a, g), y = gamma_mt(b, g);
        return x / (x + y);
    }
    const double la = log_gamma_unit(a, g), lb = log_gamma_unit(b, g);   // x / (x + y) = inv_logit(log x - log y)
    const double t = la - lb;
    return t >= 0.0 ? 1.0 / (1.0 + exp(-t)) : exp(t) / (1.0 + exp(t));
}

SMCB_HD double student_t_rng(double nu, double mu, double sigma, Rng& g) {
    if (!(positive(nu) && finite(mu) && positive(sigma))) return g.fail();
    const double z = std_normal_rng(g);
    const double chi2 = 2.0 * gamma_unit(0.5 * nu, g);
    return mu + sigma * z / sqrt(chi2 / nu);
}

// ---- discrete (values are integers, returned as doubles)
SMCB_HD double bernoulli_rng(double p, Rng& g) {
    if (!(p >= 0.0 && p <= 1.0)) return g.fail();
    return g.unit() < p ? 1.0 : 0.0;
}

SMCB_HD double bernoulli_logit_rng(double eta, Rng& g) {
    if (eta != eta) return g.fail();
    const double e = exp(-fabs(eta)), p = eta >= 0.0 ? 1.0 / (1.0 + e) : e / (1.0 + e);
    return g.unit() < p ? 1.0 : 0.0;
}

SMCB_HD double poisson_rng(double lam, Rng& g) {
    if (!(lam >= 0.0 && lam < kPoissonMaxRate)) return g.fail();
    if (lam == 0.0) return 0.0;
    if (lam < 10.0) {                        // inversion: the smallest k with u < F(k)
        double p = exp(-lam), s = p, k = 0.0;
        const double u = g.unit();
        while (u >= s && k < 400.0) {
            k += 1.0;
            p *= lam / k;
            s += p;
        }
        return k;
    }
    // PTRS: W. Hoermann, "The transformed rejection method for generating Poisson random variables" (1993)
    const double slam = sqrt(lam), loglam = log(lam);
    const double b = 0.931 + 2.53 * slam, a = -0.059 + 0.02483 * b;
    const double log_invalpha = log(1.1239 + 1.1328 / (b - 3.4)), vr = 0.9277 - 3.6224 / (b - 2.0);
    for (int it = 0; it < kMaxTrials; ++it) {
        const double u = g.open() - 0.5, v = g.open();
        const double us = 0.5 - fabs(u);
        const double k = floor((2.0 * a / us + b) * u + lam + 0.43);
        if (us >= 0.07 && v <= vr) return k;
        if (k < 0.0 || (us < 0.013 && v > us)) continue;
        if (log(v) + log_invalpha - log(a / (us * us) + b) <= -lam + k * loglam - lgamma(k + 1.0)) return k;
    }
    return g.fail();
}

SMCB_HD double poisson_log_rng(double eta, Rng& g) {
    if (!(eta < log(kPoissonMaxRate))) return g.fail();
    return poisson_rng(exp(eta), g);
}

SMCB_HD double binomial_rng(double n, double p, Rng& g) {
    if (!(n >= 0.0 && n <= 2147483647.0 && n == floor(n) && p >= 0.0 && p <= 1.0)) return g.fail();
    if (n == 0.0 || p == 0.0) return 0.0;
    if (p == 1.0) return n;
    const bool flip = p > 0.5;
    const double pp = flip ? 1.0 - p : p, q = 1.0 - pp;
    double k = NAN;
    if (n * pp < 10.0) {                     // inversion, restarted when it walks past a far bound (numpy's)
        const double qn = exp(n * log1p(-pp)), r = pp / q;
        const double bound = fmin(n, n * pp + 10.0 * sqrt(n * pp * q + 1.0));
        for (int it = 0; it < kMaxTrials && !(k == k); ++it) {
            double x = 0.0, px = qn, u = g.unit();
            while (u > px && x <= bound) {
                x += 1.0;
                u -= px;
                px *= (n - x + 1.0) * r / x;
            }
            if (x <= bound) k = x;
        }
    } else {
        // BTRS: W. Hoermann, "The generation of binomial random variates" (1993); the acceptance test against the exact
        // log ratio of the pmf at k and at the mode m
        const double spq = sqrt(n * pp * q);
        const double b = 1.15 + 2.53 * spq, a = -0.0873 + 0.0248 * b + 0.01 * pp, c = n * pp + 0.5;
        const double vr = 0.92 - 4.2 / b, alpha = (2.83 + 5.1 / b) * spq, lpq = log(pp / q);
        const double m = floor((n + 1.0) * pp), hm = lgamma(m + 1.0) + lgamma(n - m + 1.0);
        for (int it = 0; it < kMaxTrials; ++it) {
            const double u = g.open() - 0.5, v = g.open();
            const double us = 0.5 - fabs(u);
            const double kk = floor((2.0 * a / us + b) * u + c);
            if (kk < 0.0 || kk > n) continue;
            if (us >= 0.07 && v <= vr) {
                k = kk;
                break;
            }
            if (log(v * alpha / (a / (us * us) + b)) <= hm - lgamma(kk + 1.0) - lgamma(n - kk + 1.0) + (kk - m) * lpq) {
                k = kk;
                break;
            }
        }
    }
    if (!(k == k)) return g.fail();
    return flip ? n - k : k;
}

SMCB_HD double neg_binomial_2_rng(double mu, double phi, Rng& g) {
    if (!(positive(mu) && positive(phi))) return g.fail();
    const double lam = gamma_unit(phi, g) * (mu / phi);
    if (!(lam < kPoissonMaxRate)) return g.fail();
    return poisson_rng(lam, g);
}

// theta: a simplex (entries >= 0, sum within 1e-8 of 1) -> 1 .. K
template <int K>
SMCB_HD double categorical_rng(const double* theta, Rng& g) {
    double s = 0.0;
    bool valid = true;
    for (int k = 0; k < K; ++k) {
        valid = valid && theta[k] >= 0.0;
        s += theta[k];
    }
    if (!(valid && fabs(s - 1.0) <= 1e-8)) return g.fail();
    const double u = g.unit();
    double c = 0.0;
    for (int k = 0; k < K - 1; ++k) {
        c += theta[k];
        if (u < c) return k + 1.0;
    }
    return (double)K;
}

}  // namespace stan
}  // namespace smcb
