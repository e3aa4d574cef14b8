// K1 -- fused tempered log-posterior + gradient device functions.
//
// Replaces the per-particle BridgeStan calls of /root/reference/smcnuts/model/bridgestan.py:28-90
// (log_density / log_density_gradient, one ctypes call per particle per leapfrog, and a JSON rewrite +
// model reload per phi change, :122-146).  Every model returns the split
//     logp(x, phi) = A(x) + phi * B(x),   A = log prior + log Jacobian,  B = log likelihood
// (the identity adaptive_tempering.py:38-43 relies on), so phi is a plain kernel argument and one
// evaluation serves NUTS (at phi_new), the phi=1 reweight (samples.py:190-191) and the tempering
// bisection (adaptive_tempering.py:38-39) at once.
//
//   ArmaModel   /root/reference/stan_models/arma/arma.stan:16-30        x = (mu, beta, theta, log sigma)
//   PrmModel    /root/reference/stan_models/PRMwCD/PRMwCD.stan:17-39    x = (Beta_1..12, log Gamma)
//   GaussModel  synthetic correlated Gaussian of BASELINE.json config 4 (SURVEY.md section 8d)
//
// Arithmetic order follows oracle/smc_oracle.c statement by statement (device FMA contraction is the
// only difference), so device and oracle agree to ~1e-15 relative.
#pragma once
#include "common.cuh"

// Warp-level code (shuffles, votes, mma.sync) is compiled for the device and, with SMCB_SIMT_EMU, for the fiber-based
// warp emulator of tests/hostsim (a test tool that runs the 4-lanes-per-particle kernels on the CPU; never part of the
// product library).
#if defined(__CUDA_ARCH__) || defined(SMCB_SIMT_EMU)
#define SMCB_WARP_CODE 1
#endif

namespace smcb {

#if defined(SMCB_WARP_CODE)
// C[8x8] += A[8x4] * B[4x8] on FP64 tensor cores; per-lane fragments: A[l/4][l%4], B[l%4][l/4], C[l/4][2(l%4) + {0,1}]
SMCB_D void dmma(double& c0, double& c1, double a, double b) {
#if defined(__CUDA_ARCH__)
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
#else
    simt_emu::dmma(c0, c1, a, b);
#endif
}
#endif

// Plain-old-data descriptor handed to kernels by value; `data` points at the packed device blob.
struct ModelDesc {
    int kind;
    int dim;
    int n_data;          // doubles in `data`
    int T;               // arma: series length; PRMwCD: number of observations
    double q;            // PRMwCD: exponent of the exponential-power prior
    const double* data;  // device (or, in tests/hostsim, host) pointer
    const double* scale; // [dim] diagonal metric (nullable): NUTS then runs on z = x / scale (ScaledModel below)
};

// ---------------------------------------------------------------------------------------------- arma
#ifndef SMCB_ARMA_UNROLL
#define SMCB_ARMA_UNROLL 8     // A/B on B200 (profiles/r2_ab_arma_unroll.log)
#endif
constexpr int kArmaUnroll = SMCB_ARMA_UNROLL;
struct ArmaModel {
    static constexpr int DMAX = 4;
    static constexpr int STATIC_D = 4;
    static constexpr int GROUP = 1, NLOC = 4, STATIC_NL = 4;   // one lane per particle, 4 coordinates per lane
    static constexpr bool STAGE = false;                       // U-turn operands straight from the workspace (see nuts_lane.cuh)
    SMCB_HD constexpr int nloc() const { return 4; }
    const double* y;
    int T;
    SMCB_HD explicit ArmaModel(const ModelDesc& d, const double* staged) : y(staged), T(d.T) {}
    SMCB_HD static constexpr int dim_of(const ModelDesc&) { return 4; }
    SMCB_HD constexpr int dim() const { return 4; }
    static int staged_doubles(const ModelDesc& d) { return d.T; }

    // A, B and g = grad A + phi * grad B
    SMCB_HD void eval(const double (&x)[DMAX], double phi, double& A, double& B, double (&g)[DMAX]) const {
        const double mu = x[0], beta = x[1], theta = x[2], s = x[3];
#if SMCB_FAST_PATH
        // Device fast path of the prior block (same formulas, a few ulp apart from the host/oracle statement order):
        // sigma^2 and 1/sigma^2 from one interleaved exp pair instead of exp + multiply + divide, divisions by
        // constants as multiplications, one division shared by the Cauchy gradient.  The whole block is ~12 % of the
        // NUTS kernel's warp time when done with libm calls and four divisions.
        double sig2, inv;
        fast_exp_pair(2.0 * s, -2.0 * s, sig2, inv);
        const double q = sig2 * 0.16;
        const double cauchy_g = 2.0 * q / (1.0 + q);
        const bool sigma_ok = (s > -745.13321910194122) && (s < 709.78271289338397);   // exp(s) finite and > 0
        A = (-0.5 * kLog2Pi - 2.3025850929940456840 - mu * mu * 0.005) +
            (-0.5 * kLog2Pi - 0.69314718055994530942 - beta * beta * 0.125) +
            (-0.5 * kLog2Pi - 0.69314718055994530942 - theta * theta * 0.125) +
            (-kLogPi - 0.91629073187415506518 - fast_log(1.0 + q)) + s;
#else
        // the oracle's statement order (oracle/smc_oracle.c::arma_split): host builds and the parity device build
        const double sigma = fast_exp(s), sig2 = sigma * sigma, q = sig2 / 6.25;
        const double inv = 1.0 / sig2;
        const double cauchy_g = 2.0 * q / (1.0 + q);
        const bool sigma_ok = is_finite(sigma) && sigma > 0.0;
        A = (-0.5 * kLog2Pi - 2.3025850929940456840 - mu * mu / 200.0) +
            (-0.5 * kLog2Pi - 0.69314718055994530942 - beta * beta / 8.0) +
            (-0.5 * kLog2Pi - 0.69314718055994530942 - theta * theta / 8.0) +
            (-kLogPi - 0.91629073187415506518 - ref_log1p(q)) + s;
#endif
        double ylag = y[0];
        double e = ylag - (mu + beta * mu);
        double dm = -(1.0 + beta), db = -mu, dt = 0.0;
        double S = e * e, Sm = e * dm, Sb = e * db, St = e * dt;
        // One DFMA per loop-carried chain and step (e, d_mu, d_beta, d_theta) plus four accumulator DFMAs: the
        // y-only part of nu[t] is formed off the critical path, so a single warp keeps the FP64 pipe busy.
        const double ntheta = -theta;
#pragma unroll kArmaUnroll
        for (int t = 1; t < T; ++t) {
            const double yt = y[t];
            const double c = yt - (mu + beta * ylag);       // y[t] - (mu + beta*y[t-1]); independent of the chains
            const double en = ntheta * e + c;                // err[t] = y[t] - nu[t]              (arma.stan:26-27)
            const double dmn = ntheta * dm - 1.0;
            const double dbn = ntheta * db - ylag;
            const double dtn = ntheta * dt - e;
            e = en; dm = dmn; db = dbn; dt = dtn; ylag = yt;
            S += e * e; Sm += e * dm; Sb += e * db; St += e * dt;
        }
        B = -0.5 * T * kLog2Pi - T * s - 0.5 * S * inv;
        if (!sigma_ok) A = neg_inf();
#if SMCB_FAST_PATH
        g[0] = -mu * 0.01 + phi * (-Sm * inv);
#else
        g[0] = -mu / 100.0 + phi * (-Sm * inv);
#endif
        g[1] = -beta / 4.0 + phi * (-Sb * inv);
        g[2] = -theta / 4.0 + phi * (-St * inv);
        g[3] = (1.0 - cauchy_g) + phi * (-T + S * inv);
    }
};

// ---------------------------------------------------------------------------------------------- PRMwCD
// Packed device layout (built by smcb_model_create from the host blob [q, y(NO), lgamma(y+1)(NO), X(NO x 11)]):
//   header, 16 doubles: [0] sum_i y_i, [1..11] (X'y)_j, [12] sum_i lgamma(y_i+1), [13..15] 0
//   per observation i, 12 doubles: X_i0..X_i10, y_i                                   -> 16-byte aligned rows
// With the y-weighted sums hoisted, sum_i [y_i eta_i - exp(eta_i) - lgamma(y_i+1)] needs only exp(eta_i) and
// 11 FMAs per observation for the gradient (PRMwCD.stan:24-33), two shorter eta chains instead of one.
// Exponential-power prior term of one coefficient (PRMwCD.stan:36-37): aq = |b / Gamma|^q and d(-aq)/db = -q aq / b.
// Device fast path for q = 1/2: with sg = Gamma^(-1/2) and r = rsqrt(|b|), aq = sg |b| r and aq / b = sg r sign(b): one
// rsqrt instead of sqrt + divide (a few ulp apart from the host/oracle form).
SMCB_HD void prm_prior_term(double b, double q, double ig, double sg, double& aq, double& dterm) {
#if SMCB_FAST_PATH
    if (q == 0.5) {
        const double ab = fabs(b), r = rsqrt(ab);
        aq = (ab == 0.0) ? 0.0 : sg * ab * r;
        dterm = -0.5 * sg * copysign(r, b);
        (void)ig;
        return;
    }
#endif
    (void)sg;
    const double a = fabs(b) * ig;
    aq = (q == 0.5) ? sqrt(a) : pow(a, q);
    dterm = -q * aq / b;
}
// Gamma^-1 and Gamma^-1/2 from log Gamma; finite, positive Gamma <=> exp(gg) neither overflows nor underflows
SMCB_HD void prm_gamma_terms(double gg, double& ig, double& sg, bool& ok) {
#if SMCB_FAST_PATH
    sg = fast_exp(-0.5 * gg);
    ig = sg * sg;
    ok = (gg > -745.13321910194122) && (gg < 709.78271289338397);
#else
    ig = fast_exp(-gg);
    sg = 0.0;
    const double Gam = fast_exp(gg);
    ok = is_finite(Gam) && Gam > 0.0;
#endif
}

struct PrmModel {
    static constexpr int DMAX = 13;
    static constexpr int STATIC_D = 13;
    static constexpr int GROUP = 1, NLOC = 13, STATIC_NL = 13;
    static constexpr bool STAGE = false;
    SMCB_HD constexpr int nloc() const { return 13; }
    static constexpr int M = 12, C = 11, ROW = 12, HDR = 16;
    const double* hdr;
    const double* rows;
    int NO;
    double q;
    SMCB_HD explicit PrmModel(const ModelDesc& d, const double* staged) : hdr(staged), rows(staged + HDR), NO(d.T), q(d.q) {}
    SMCB_HD static constexpr int dim_of(const ModelDesc&) { return 13; }
    SMCB_HD constexpr int dim() const { return 13; }
    static int staged_doubles(const ModelDesc& d) { return HDR + d.T * ROW; }

    SMCB_HD void eval(const double (&x)[DMAX], double phi, double& A, double& B, double (&g)[DMAX]) const {
        const double gg = x[M];
        double slam = 0.0, min_eta = 1e308;
        double gl[M];   // sum_i lambda_i * (1, X_i.)
#pragma unroll
        for (int j = 0; j < M; ++j) gl[j] = 0.0;
        // observations two at a time with their dependency chains interleaved (eta: 4 chains; exp: 2 x 2 chains)
        int i = 0;
#pragma unroll 1
        for (; i + 1 < NO; i += 2) {
            const double* rowa = rows + i * ROW;
            const double* rowb = rowa + ROW;
            double xa_[C], xb_[C];
#pragma unroll
            for (int j = 0; j < C; ++j) { xa_[j] = rowa[j]; xb_[j] = rowb[j]; }
            double a0 = x[0], a1 = 0.0, b0 = x[0], b1 = 0.0;
#pragma unroll
            for (int j = 0; j < C; j += 2) {
                a0 += x[j + 1] * xa_[j];
                b0 += x[j + 1] * xb_[j];
                if (j + 1 < C) {
                    a1 += x[j + 2] * xa_[j + 1];
                    b1 += x[j + 2] * xb_[j + 1];
                }
            }
            const double etaa = a0 + a1, etab = b0 + b1;
            min_eta = etaa < min_eta ? etaa : min_eta;
            min_eta = etab < min_eta ? etab : min_eta;
            double lama, lamb;
            fast_exp_pair(etaa, etab, lama, lamb);
            slam += lama; gl[0] += lama;
#pragma unroll
            for (int j = 0; j < C; ++j) gl[j + 1] += lama * xa_[j];
            slam += lamb; gl[0] += lamb;
#pragma unroll
            for (int j = 0; j < C; ++j) gl[j + 1] += lamb * xb_[j];
        }
        for (; i < NO; ++i) {   // odd tail
            const double* row = rows + i * ROW;
            double e0 = x[0], e1 = 0.0;
#pragma unroll
            for (int j = 0; j < C; j += 2) {
                e0 += x[j + 1] * row[j];
                if (j + 1 < C) e1 += x[j + 2] * row[j + 1];
            }
            const double eta = e0 + e1;
            min_eta = eta < min_eta ? eta : min_eta;
            const double lam = fast_exp(eta);
            slam += lam; gl[0] += lam;
#pragma unroll
            for (int j = 0; j < C; ++j) gl[j + 1] += lam * row[j];
        }
        // sum_i y_i eta_i = Beta_1 sum y + sum_j Beta_{j+1} (X'y)_j
        double ydot = x[0] * hdr[0];
#pragma unroll
        for (int j = 0; j < C; ++j) ydot += x[j + 1] * hdr[1 + j];
        double b = ydot - slam - hdr[12];
        // Stan's poisson_lpmf is -inf when lambda underflows to 0 with y > 0 (and when lambda = inf: slam = inf above)
        if (fast_exp(min_eta) == 0.0) {
            for (int i = 0; i < NO; ++i) {
                const double* row = rows + i * ROW;
                double eta = x[0];
                for (int j = 0; j < C; ++j) eta += x[j + 1] * row[j];
                if (fast_exp(eta) == 0.0 && row[11] > 0.0) b = neg_inf();
            }
        }
        B = b;
        double ig, sg, sum = 0.0;
        bool gam_ok;
        prm_gamma_terms(gg, ig, sg, gam_ok);
        g[0] = phi * (hdr[0] - gl[0]);
#pragma unroll
        for (int i = 1; i < M; ++i) {
            double aq, dterm;
            prm_prior_term(x[i], q, ig, sg, aq, dterm);
            sum += aq;
            g[i] = dterm + phi * (hdr[i] - gl[i]);
        }
        A = (2.0 * 0.26236426446749105204 - 0.0 - 3.0 * gg - 1.3 * ig) + gg + (-(M - 1) * gg - sum);
        g[M] = -3.0 + 1.3 * ig + 1.0 - (M - 1) + q * sum;
        if (!gam_ok) A = neg_inf();
    }
};

// Tensor-core variant of PRMwCD for the NUTS kernel: 4 lanes per particle, 8 particles per warp (the group layout of
// GaussModelG below).  Lane `sub` of a group holds coordinates sub, sub+4, sub+8, sub+12 (coordinate 12 = log Gamma sits
// in lane 0, 13..15 are padding).  With Xt = [1, X] (NO x 12) the evaluation is two small FP64 GEMMs over 8 particles,
//     eta = Beta Xt'   (8 x 12 times 12 x NO)      lambda = exp(eta)      G = lambda Xt   (8 x NO times NO x 12)
// issued as mma.m8n8k4 (DMMA) on tiles of 8 observations: the C fragment of an eta tile (lane (g,t) holds observations
// 2t, 2t+1 of particle g) is, after the exp, directly the A fragment of two k-steps of the second product, because the
// rows of its B fragments are packed in that order; the columns of the second product are permuted so that lane t
// receives exactly the gradient entries of the coordinates it owns.  No shuffles, 7 DMMA + 2 exp per lane and tile;
// per-particle latency is ~4x shorter than one-lane-per-particle, which is what the 2047-leapfrog trees need.
// Padded observations (NO..8*NT-1) have all-zero rows in both products, so sum_i lambda_i is column 0 of G.
//
// Staged block (built by pack_prm_fragments, appended to the scalar blob):
//   [0..15]  hy: sum y, (X'y)_1..11, 0...      [16] sum lgamma(y+1)    [17..31] 0
//   pf1[NT][3][32]      B fragments of the first product  (k = 4kk + l%4, observation 8nt + l/4)
//   pf2[NT][2][2][32]   B fragments of the second product (observation 8nt + 2(l%4) + h, column 8nt2 + 4(n%2) + n/2, n = l/4)
//   ym [NT][2][32]      1.0 where that observation has y > 0 (only read on the lambda-underflow path)
template <int NT>
struct PrmModelG {
    static constexpr int DMAX = 16;
    static constexpr int STATIC_D = 0;
    static constexpr int GROUP = 4, NLOC = 4, STATIC_NL = 4;
    static constexpr bool STAGE = false;
    static constexpr int M = 12, HDRG = 32;
    static constexpr int PF1 = HDRG, PF2 = PF1 + NT * 3 * 32, YM = PF2 + NT * 4 * 32, TOTAL = YM + NT * 2 * 32;
    const double* blk;
    double q;
    SMCB_HD explicit PrmModelG(const ModelDesc& d, const double* staged) : blk(staged), q(d.q) {}
    SMCB_HD static constexpr int dim_of(const ModelDesc&) { return 13; }
    SMCB_HD constexpr int dim() const { return 13; }
    SMCB_HD constexpr int nloc() const { return NLOC; }
    static int staged_doubles(const ModelDesc&) { return TOTAL; }
    static bool fits(const ModelDesc& d) { return d.T <= 8 * NT && d.T > 8 * (NT - 3); }

#if defined(SMCB_WARP_CODE)
    // W tiles starting at the fragment pointers q1 (first product) / q2 (second product): eta, lambda = exp(eta), and
    // lambda's contribution to the two accumulator sets (tiles alternate between them to halve the DMMA chains)
    template <int W>
    static SMCB_D void tile_block(const double (&x)[NLOC], const double* q1, const double* q2,
                                                      double (&c)[2][4], unsigned& neg_hi) {
        double e[2 * W];
#pragma unroll
        for (int u = 0; u < W; ++u) { e[2 * u] = 0.0; e[2 * u + 1] = 0.0; }
#pragma unroll
        for (int kk = 0; kk < 3; ++kk) {
#pragma unroll
            for (int u = 0; u < W; ++u) dmma(e[2 * u], e[2 * u + 1], x[kk], q1[(u * 3 + kk) * 32]);
        }
        // most negative eta so far, tracked on the integer pipe: for negative doubles the high word grows (as an
        // unsigned integer) with the magnitude; positive values have the sign bit clear and never win
#pragma unroll
        for (int i = 0; i < 2 * W; ++i) neg_hi = max(neg_hi, (unsigned)__double2hiint(e[i]));
#pragma unroll
        for (int u = 0; u < W; ++u) fast_exp_pair(e[2 * u], e[2 * u + 1], e[2 * u], e[2 * u + 1]);
#pragma unroll
        for (int u = 0; u < W; ++u) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
#pragma unroll
                for (int nt2 = 0; nt2 < 2; ++nt2)
                    dmma(c[u & 1][2 * nt2], c[u & 1][2 * nt2 + 1], e[2 * u + h], q2[((u * 2 + h) * 2 + nt2) * 32]);
            }
        }
    }
#endif

    SMCB_HD void eval(const double (&x)[NLOC], double phi, double& A, double& B, double (&g)[NLOC]) const {
#if defined(SMCB_WARP_CODE)
        constexpr unsigned kFull = 0xffffffffu;
        constexpr double kExpZero = -745.13321910194122;   // exp(x) rounds to 0 below ln(2^-1075)
        const int lane = threadIdx.x & 31, sub = lane & 3;
        const double* p1 = blk + PF1 + lane;
        const double* p2 = blk + PF2 + lane;
        // ---- tiles of 8 observations in a ROLLED loop.  The kernel is instruction-fetch bound when this body is
        //      unrolled (MEASURED at N = 2^20, 4 CTAs/SM: all 13 tiles unrolled 190 ms with `no_instruction` 3.3 stalls
        //      per issue; 6 tiles per trip 153 ms; 4: 140 ms; 2: 132 ms; 1: 130.5 ms): with four warps per scheduler at
        //      different places of a large kernel, the small loop body is what stays in the instruction cache, and the
        //      other warps supply the parallelism that unrolling would have.
        double c[2][4];
#pragma unroll
        for (int a_ = 0; a_ < 2; ++a_)
#pragma unroll
            for (int i = 0; i < 4; ++i) c[a_][i] = 0.0;
        unsigned neg_hi = 0u;
        constexpr int U = 1;
        int nt0 = 0;
#pragma unroll 1
        for (; nt0 + U <= NT; nt0 += U) tile_block<U>(x, p1 + nt0 * 96, p2 + nt0 * 128, c, neg_hi);
        if constexpr (NT % U != 0) tile_block<NT % U>(x, p1 + nt0 * 96, p2 + nt0 * 128, c, neg_hi);
        double gl[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) gl[i] = c[0][i] + c[1][i];
        // ---- group scalars: log Gamma lives in slot 3 of lane 0, sum lambda in slot 0 of lane 0
        const int first = lane & ~3;
        const double gg = __shfl_sync(kFull, x[3], first);
        const double slam = __shfl_sync(kFull, gl[0], first);
        neg_hi = max(neg_hi, __shfl_xor_sync(kFull, neg_hi, 1));
        neg_hi = max(neg_hi, __shfl_xor_sync(kFull, neg_hi, 2));
        double ig, sg;
        bool gam_ok;
        prm_gamma_terms(gg, ig, sg, gam_ok);
        double ydot = 0.0, sum = 0.0;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const int j = sub + 4 * i;           // coordinates 0..11
            const double hyj = blk[j];
            ydot += x[i] * hyj;
            if (j == 0) {
                g[i] = phi * (hyj - gl[i]);
            } else {
                double aq, dterm;
                prm_prior_term(x[i], q, ig, sg, aq, dterm);
                sum += aq;
                g[i] = dterm + phi * (hyj - gl[i]);
            }
        }
        ydot += __shfl_xor_sync(kFull, ydot, 1); sum += __shfl_xor_sync(kFull, sum, 1);
        ydot += __shfl_xor_sync(kFull, ydot, 2); sum += __shfl_xor_sync(kFull, sum, 2);
        g[3] = (sub == 0) ? (-3.0 + 1.3 * ig + 1.0 - (M - 1) + q * sum) : 0.0;
        double b = ydot - slam - blk[16];
        // Stan's poisson_lpmf is -inf when lambda underflows to 0 with y > 0 (warp-uniform slow path: the DMMAs need
        // every lane); lambda = inf gives slam = inf or, through a zero entry of Xt, NaN -> -inf as well
        // high word of kExpZero with the sign bit: a (slightly conservative) trigger, the slow path compares exactly
        if (__any_sync(kFull, neg_hi >= 0xc0874910u)) {
            __syncwarp();
            bool hit = false;
            const double* pm = blk + YM + lane;
#pragma unroll 1
            for (int nt = 0; nt < NT; ++nt) {
                double e0 = 0.0, e1 = 0.0;
#pragma unroll
                for (int kk = 0; kk < 3; ++kk) dmma(e0, e1, x[kk], p1[(nt * 3 + kk) * 32]);
                hit |= (e0 < kExpZero && pm[(nt * 2) * 32] > 0.0) || (e1 < kExpZero && pm[(nt * 2 + 1) * 32] > 0.0);
            }
            const unsigned hits = __ballot_sync(kFull, hit);
            if ((hits >> first) & 0xfu) b = neg_inf();
        }
        if (b != b) b = neg_inf();
        B = b;
        A = (2.0 * 0.26236426446749105204 - 0.0 - 3.0 * gg - 1.3 * ig) + gg + (-(M - 1) * gg - sum);
        if (!gam_ok) A = neg_inf();
#else
        (void)x; (void)phi; A = B = 0.0; (void)g;
#endif
    }
};

// host-side packing of the staged block of PrmModelG from the scalar blob (PrmModel layout: header + NO rows of 12)
inline void pack_prm_fragments(const double* scalar_blob, int NO, int nt_tiles, double* out) {
    const double* hdr = scalar_blob;
    const double* rows = scalar_blob + 16;
    auto xt = [&](int o, int k) -> double {   // Xt = [1, X], zero outside the data
        if (o >= NO || k >= 12) return 0.0;
        return k == 0 ? 1.0 : rows[(size_t)o * 12 + (k - 1)];
    };
    const int PF1 = 32, PF2 = PF1 + nt_tiles * 3 * 32, YM = PF2 + nt_tiles * 4 * 32;
    for (int i = 0; i < 32; ++i) out[i] = 0.0;
    for (int j = 0; j < 12; ++j) out[j] = hdr[j];
    out[16] = hdr[12];
    for (int nt = 0; nt < nt_tiles; ++nt)
        for (int l = 0; l < 32; ++l) {
            for (int kk = 0; kk < 3; ++kk) out[PF1 + (nt * 3 + kk) * 32 + l] = xt(8 * nt + l / 4, 4 * kk + l % 4);
            for (int h = 0; h < 2; ++h) {
                const int o = 8 * nt + 2 * (l % 4) + h, n = l / 4;
                for (int nt2 = 0; nt2 < 2; ++nt2)
                    out[PF2 + ((nt * 2 + h) * 2 + nt2) * 32 + l] = xt(o, 8 * nt2 + 4 * (n % 2) + n / 2);
                out[YM + (nt * 2 + h) * 32 + l] = (o < NO && rows[(size_t)o * 12 + 11] > 0.0) ? 1.0 : 0.0;
            }
        }
}

// ---------------------------------------------------------------------------------------------- Gaussian
// data = P (D x D row-major, symmetric).  A = 0, B = -x'Px/2, grad B = -P x.  One thread per particle,
// state in local memory (runtime D <= DMAX); P is read through L1/L2 (all lanes read the same address).
struct GaussModel {
    static constexpr int DMAX = 128;
    static constexpr int STATIC_D = 0;  // runtime dimension
    static constexpr int GROUP = 1, NLOC = 128, STATIC_NL = 0;
    static constexpr bool STAGE = false;
    SMCB_HD int nloc() const { return D; }
    const double* P;
    int D;
    SMCB_HD explicit GaussModel(const ModelDesc& d, const double* staged) : P(staged), D(d.dim) {}
    SMCB_HD static int dim_of(const ModelDesc& d) { return d.dim; }
    SMCB_HD int dim() const { return D; }
    static int staged_doubles(const ModelDesc&) { return 0; }  // too large for smem at D = 100 with state; use L1/L2

    SMCB_HD void eval(const double (&x)[DMAX], double phi, double& A, double& B, double (&g)[DMAX]) const {
        double qf = 0.0;
        for (int i = 0; i < D; ++i) {
            double acc = 0.0;
            const double* row = P + (size_t)i * D;
#pragma unroll 4
            for (int k = 0; k < D; ++k) acc += row[k] * x[k];
            g[i] = phi * (-acc);
            qf += x[i] * acc;
        }
        A = 0.0;
        B = -0.5 * qf;
    }
};

// Tensor-core variant for the NUTS kernel: 4 lanes per particle, 8 particles per warp.  Lane `sub` of a group holds
// coordinates sub, sub+4, ... (exactly the A-fragment layout of mma.m8n8k4: row = particle, col = k), the precision
// matrix is pre-packed on the host in B-fragment order with the columns of every 8-block permuted so that the C
// fragment lands in the same ownership pattern (no shuffles): -P x for 8 particles costs 2*NT8^2 DMMA + as many
// conflict-free 256-byte shared-memory loads.  NT8 = ceil(D/8) blocks of 8 coordinates (zero padded).
template <int NT8>
struct GaussModelG {
    static constexpr int DMAX = 8 * NT8;
    static constexpr int STATIC_D = 0;
    static constexpr int GROUP = 4, NLOC = 2 * NT8, STATIC_NL = 2 * NT8, KK = 2 * NT8;
    // wide records (> 4 coordinates per lane): the stored edge of a U-turn test is staged in shared memory (cp.async /
    // the previous leaf written directly) instead of being loaded into registers the kernel does not have
#if defined(SMCB_NO_STAGE)   // A/B experiments only
    static constexpr bool STAGE = false;
#else
    static constexpr bool STAGE = NLOC > 4;
#endif
    const double* pfrag;  // [NT8][KK][32] doubles, shared memory
    int D;
    SMCB_HD explicit GaussModelG(const ModelDesc& d, const double* staged) : pfrag(staged), D(d.dim) {}
    SMCB_HD static int dim_of(const ModelDesc& d) { return d.dim; }
    SMCB_HD int dim() const { return D; }
    SMCB_HD constexpr int nloc() const { return NLOC; }
    static int staged_doubles(const ModelDesc&) { return NT8 * KK * 32; }
    static int frag_offset(const ModelDesc& d) { return d.dim * d.dim; }  // pfrag follows the plain matrix in the blob

    SMCB_HD void eval(const double (&x)[NLOC], double phi, double& A, double& B, double (&g)[NLOC]) const {
#if defined(SMCB_WARP_CODE)
        const int lane = threadIdx.x & 31;
        // k outer, n-tiles inner: NT8 independent accumulator chains per k-step keep the tensor pipe full
        double c[NLOC];
#pragma unroll
        for (int i = 0; i < NLOC; ++i) c[i] = 0.0;
        const double* bp = pfrag + lane;
#pragma unroll
        for (int kk = 0; kk < KK; ++kk) {
            const double av = x[kk];
#pragma unroll
            for (int nt = 0; nt < NT8; ++nt) {
                dmma(c[2 * nt], c[2 * nt + 1], av, bp[(nt * KK + kk) * 32]);
            }
        }
        double qf = 0.0, qf1 = 0.0;   // two partial sums: the NLOC-term chain of dependent DFMAs is pure latency
#pragma unroll
        for (int i = 0; i < NLOC; i += 2) {
            g[i] = phi * (-c[i]);
            qf += x[i] * c[i];
            g[i + 1] = phi * (-c[i + 1]);
            qf1 += x[i + 1] * c[i + 1];
        }
        qf += qf1;
        qf += __shfl_xor_sync(0xffffffffu, qf, 1);
        qf += __shfl_xor_sync(0xffffffffu, qf, 2);
        A = 0.0;
        B = -0.5 * qf;
#else
        (void)x; (void)phi; A = B = 0.0; (void)g;
#endif
    }
};

// host-side packing of P into B-fragment order (see GaussModelG)
inline void pack_gauss_fragments(const double* P, int D, int nt8, double* out) {
    const int KK = 2 * nt8;
    for (int nt = 0; nt < nt8; ++nt)
        for (int kk = 0; kk < KK; ++kk)
            for (int l = 0; l < 32; ++l) {
                const int k = 4 * kk + (l % 4);
                const int n = l / 4;
                const int col = 8 * nt + 4 * (n % 2) + n / 2;
                out[((size_t)nt * KK + kk) * 32 + l] = (k < D && col < D) ? P[(size_t)k * D + col] : 0.0;
            }
}

// ---------------------------------------------------------------------------------------------- diagonal metric
// NUTS with a diagonal mass matrix M = diag(1 / scale^2) is NUTS with the identity metric on z = x / scale:
// pi_z(z) = pi_x(scale * z) up to a constant, grad_z = scale * grad_x.  Wrapping the model keeps the lane code (leapfrog,
// U-turn test, kinetic energy with standard-normal momenta) untouched; A and B stay the x-space split log density.
// The reference's mass matrix is the identity (nuts.py:162-175); README.md:66-67 lists mass-matrix adaptation under
// future updates.  Instantiated only for the opt-in path (csrc/nuts_kernel_scaled.cu).
template <class M>
struct ScaledModel : M {
    const double* scale;
    int d_;
    SMCB_HD explicit ScaledModel(const ModelDesc& d, const double* staged) : M(d, staged), scale(d.scale), d_(d.dim) {}
    SMCB_HD void eval(const double (&z)[M::NLOC], double phi, double& A, double& B, double (&g)[M::NLOC]) const {
        double x[M::NLOC], s[M::NLOC];
#if defined(SMCB_WARP_CODE)   // the device, and the warp emulator of tests/hostsim: lane `sub` of a group
        const int sub = (M::GROUP == 1) ? 0 : (int)(threadIdx.x % M::GROUP);
#else
        const int sub = 0;
#endif
        const int n = M::STATIC_NL ? M::STATIC_NL : this->nloc();
#pragma unroll
        for (int i = 0; i < (M::STATIC_NL ? M::STATIC_NL : n); ++i) {
            const int c = (M::GROUP == 1) ? i : sub + M::GROUP * i;
            s[i] = (c < d_) ? SMCB_LDG(&scale[c]) : 1.0;
            x[i] = mul_rn(z[i], s[i]);
        }
        // mul_rn: with plain products nvcc is free to fuse them with the model's arithmetic, and it compiles the
        // wrapped model differently from the unwrapped one (arma: 178 DMUL in the kernel against 166 with mul_rn, same
        // DFMA count, a different schedule; the differing instruction was not traced).  MEASURED on B200: scale = ones
        // then left x_new 1 ulp away from the identity-metric kernel in 122 of 2061 one-lane PRMwCD rows; with mul_rn the
        // two agree bit for bit at every dispatch tests/test_metric_kernels.py runs.
        M::eval(x, phi, A, B, g);
#pragma unroll
        for (int i = 0; i < (M::STATIC_NL ? M::STATIC_NL : n); ++i) g[i] = mul_rn(g[i], s[i]);
    }
};

}  // namespace smcb
