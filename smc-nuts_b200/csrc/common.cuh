// Common macros for the smcnuts B200 kernels.
//
// Every header under csrc/ that holds algorithm logic (philox.cuh, models.cuh, nuts_lane.cuh) is written
// against SMCB_HD so that the SAME source also compiles with plain g++ for tests/hostsim (a CPU
// simulation of the device lanes used only by the `not gpu` test-suite to validate kernel logic against
// the oracle; it is not part of, nor reachable from, the product library).
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#define SMCB_HD __host__ __device__ __forceinline__
#define SMCB_D __device__ __forceinline__
#else
#define SMCB_HD inline
#define SMCB_D inline
#endif

// Build flavours of the arithmetic (see DESIGN.md section 6):
//   product device code      SMCB_FAST_PATH = 1: fused fast paths of the prior blocks, FMA contraction by nvcc
//   parity device build      -DSMCB_PARITY=1 -fmad=false (libsmcnuts_b200_parity.so): the oracle's statement order, no
//                            contraction; exp / log are the table-driven fast_exp / fast_log below, whose explicit FMAs
//                            are reproducible on a CPU
//   host, -DSMCB_DEVMATH     tests/hostsim only: the same fast_exp / fast_log arithmetic restated for the host, so the
//                            g++ build of the lane code is the bit-for-bit twin of the parity device build
//   host, default            std::exp / std::log / log1p: bit-identical to the default oracle (glibc)
#if !defined(SMCB_PARITY)
#define SMCB_PARITY 0
#endif
#if defined(__CUDA_ARCH__) && !SMCB_PARITY
#define SMCB_FAST_PATH 1
#else
#define SMCB_FAST_PATH 0
#endif
#if defined(__CUDA_ARCH__) || defined(SMCB_DEVMATH)
#define SMCB_TABLE_MATH 1
#else
#define SMCB_TABLE_MATH 0
#endif

namespace smcb {

// bit-level access to a double, device intrinsics or (host) memcpy
SMCB_HD int dbl_hi(double v) {
#if defined(__CUDA_ARCH__)
    return __double2hiint(v);
#else
    uint64_t b; std::memcpy(&b, &v, 8); return (int)(uint32_t)(b >> 32);
#endif
}
SMCB_HD int dbl_lo(double v) {
#if defined(__CUDA_ARCH__)
    return __double2loint(v);
#else
    uint64_t b; std::memcpy(&b, &v, 8); return (int)(uint32_t)b;
#endif
}
SMCB_HD double dbl_make(int hi, int lo) {
#if defined(__CUDA_ARCH__)
    return __hiloint2double(hi, lo);
#else
    const uint64_t b = ((uint64_t)(uint32_t)hi << 32) | (uint32_t)lo; double v; std::memcpy(&v, &b, 8); return v;
#endif
}
#if defined(__CUDA_ARCH__)
#define SMCB_LDG(p) __ldg(p)
#else
#define SMCB_LDG(p) (*(p))
#endif

constexpr double kLog2Pi = 1.8378770664093454835606594728112;
constexpr double kLogPi = 1.1447298858494001741434273513531;
constexpr double kTwoPi = 6.283185307179586476925286766559;

SMCB_HD int popc32(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return __popc(v);
#else
    return __builtin_popcount(v);
#endif
}
// index of lowest set bit, v != 0
SMCB_HD int ctz32(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return __ffs((int)v) - 1;
#else
    return __builtin_ctz(v);
#endif
}
// a * b rounded on its own: never contracted into an FMA with a neighbouring addition
SMCB_HD double mul_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
SMCB_HD double neg_inf() {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double(0xfff0000000000000ULL);
#else
    return -INFINITY;
#endif
}
SMCB_HD bool is_finite(double v) {
#if defined(__CUDA_ARCH__)
    return isfinite(v);
#else
    return std::isfinite(v);
#endif
}

// exp() for the hot loops (PRMwCD: one per observation per leapfrog; log-sum-exp / normalise: one per particle).
// Table-driven: x = (32 k + j) ln2/32 + r with |r| <= ln2/64, exp(x) = 2^k * T[j] * (1 + q(r)), T[j] = 2^(j/32) from a
// 256-byte table (two L1 lines, fetched while the polynomial runs) and q = exp(r) - 1 a degree-6 Taylor polynomial in
// Estrin form: 12 FP64-pipe instructions with a 7-deep dependency chain, against 19 / 12-deep for the table-free
// degree-13 version this replaces and ~25 for libdevice's exp -- the FP64 pipe is the bound of the PRMwCD kernels,
// 35 % of whose pipe time was exp.  Max error 0.97 ulp (tests/test_gpu_parity.py checks <= 1.5 ulp against mpmath).
// For |x| < 708 (one integer compare on the high word, which also catches inf and nan) the result is a normal number
// and 2^k is applied by adding k to the exponent field: no FP64 compares, selects or scaling multiplications on the
// hot path.  Everything else takes the rare out-of-line tail: two exact scaling steps so that overflow and gradual
// underflow come out of the multiplications themselves.  Host builds (tests/hostsim) use std::exp so that they stay
// bit-identical to the oracle.
#if defined(__CUDACC__)
#define SMCB_TABLE static __device__ const double
#else
#define SMCB_TABLE static const double
#endif
#if defined(__CUDACC__) || defined(SMCB_DEVMATH)
SMCB_TABLE kExpT[32] = {
    0x1.0000000000000p+0, 0x1.059b0d3158574p+0, 0x1.0b5586cf9890fp+0, 0x1.11301d0125b51p+0, 0x1.172b83c7d517bp+0,
    0x1.1d4873168b9aap+0, 0x1.2387a6e756238p+0, 0x1.29e9df51fdee1p+0, 0x1.306fe0a31b715p+0, 0x1.371a7373aa9cbp+0,
    0x1.3dea64c123422p+0, 0x1.44e086061892dp+0, 0x1.4bfdad5362a27p+0, 0x1.5342b569d4f82p+0, 0x1.5ab07dd485429p+0,
    0x1.6247eb03a5585p+0, 0x1.6a09e667f3bcdp+0, 0x1.71f75e8ec5f74p+0, 0x1.7a11473eb0187p+0, 0x1.82589994cce13p+0,
    0x1.8ace5422aa0dbp+0, 0x1.93737b0cdc5e5p+0, 0x1.9c49182a3f090p+0, 0x1.a5503b23e255dp+0, 0x1.ae89f995ad3adp+0,
    0x1.b7f76f2fb5e47p+0, 0x1.c199bdd85529cp+0, 0x1.cb720dcef9069p+0, 0x1.d5818dcfba487p+0, 0x1.dfc97337b9b5fp+0,
    0x1.ea4afa2a490dap+0, 0x1.f50765b6e4540p+0};
constexpr int kExpFastHi = 0x40862000;            // high word of 708.0
constexpr double kExpInvL = 0x1.71547652b82fep+5;  // 32 / ln 2
constexpr double kExpLHi = 0x1.62e42fef80000p-6;   // ln 2 / 32, 34 significant bits (k' * hi is exact)
constexpr double kExpLLo = 0x1.1cf79abc9e3b4p-41;
constexpr double kExpMagic = 6755399441055744.0;   // 1.5 * 2^52: the low word of x/L + magic is round(x/L)

// p * 2^k for out-of-range arguments (|x| >= 708, inf, nan); p = T[j] exp(r) of the reduced argument
#if defined(__CUDACC__)
static __device__ __noinline__
#else
static inline
#endif
double fast_exp_tail(double x, double p, int k) {
    const int k1 = k >> 1, k2 = k - k1;
    double res = p * dbl_make((k1 + 1023) << 20, 0) * dbl_make((k2 + 1023) << 20, 0);
    res = (x > 709.782712893384) ? dbl_make(0x7ff00000, 0) : res;
    res = (x < -745.2) ? 0.0 : res;
    return (x != x) ? x : res;
}
SMCB_HD double fast_exp_scale(double p, int k) {
    return dbl_make(dbl_hi(p) + (int)((unsigned)k << 20), dbl_lo(p));
}
#endif
SMCB_HD double fast_exp(double x) {
#if SMCB_TABLE_MATH
    double t = fma(x, kExpInvL, kExpMagic);
    const int kp = dbl_lo(t);
    const double tj = SMCB_LDG(&kExpT[kp & 31]);
    t -= kExpMagic;
    double r = fma(t, -kExpLHi, x);
    r = fma(t, -kExpLLo, r);
    const double s = r * r;
    const double b0 = fma(1.0 / 6, r, 0.5);
    double b1 = fma(1.0 / 120, r, 1.0 / 24);
    b1 = fma(1.0 / 720, s, b1);
    const double q = fma(s, fma(s, b1, b0), r);
    const double p = fma(tj, q, tj);
    if ((dbl_hi(x) & 0x7fffffff) >= kExpFastHi) return fast_exp_tail(x, p, kp >> 5);
    return fast_exp_scale(p, kp >> 5);
#else
    return std::exp(x);
#endif
}

// Two independent exps with their instruction streams interleaved statement by statement (the compiler keeps the
// source order inside a basic block, so this doubles the ILP of the latency-bound chains).
SMCB_HD void fast_exp_pair(double xa, double xb, double& ea, double& eb) {
#if SMCB_TABLE_MATH
    double ta = fma(xa, kExpInvL, kExpMagic), tb = fma(xb, kExpInvL, kExpMagic);
    const int ka = dbl_lo(ta), kb = dbl_lo(tb);
    const double ja = SMCB_LDG(&kExpT[ka & 31]), jb = SMCB_LDG(&kExpT[kb & 31]);
    ta -= kExpMagic; tb -= kExpMagic;
    double ra = fma(ta, -kExpLHi, xa), rb = fma(tb, -kExpLHi, xb);
    ra = fma(ta, -kExpLLo, ra); rb = fma(tb, -kExpLLo, rb);
    const double sa = ra * ra, sb = rb * rb;
    const double a0 = fma(1.0 / 6, ra, 0.5), c0 = fma(1.0 / 6, rb, 0.5);
    double a1 = fma(1.0 / 120, ra, 1.0 / 24), c1 = fma(1.0 / 120, rb, 1.0 / 24);
    a1 = fma(1.0 / 720, sa, a1); c1 = fma(1.0 / 720, sb, c1);
    const double qa = fma(sa, fma(sa, a1, a0), ra), qb = fma(sb, fma(sb, c1, c0), rb);
    const double pa = fma(ja, qa, ja), pb = fma(jb, qb, jb);
    const int ha = dbl_hi(xa) & 0x7fffffff, hb = dbl_hi(xb) & 0x7fffffff;
    ea = fast_exp_scale(pa, ka >> 5); eb = fast_exp_scale(pb, kb >> 5);
    if ((ha > hb ? ha : hb) >= kExpFastHi) {   // rare: out-of-range, inf or nan argument
        if (ha >= kExpFastHi) ea = fast_exp_tail(xa, pa, ka >> 5);
        if (hb >= kExpFastHi) eb = fast_exp_tail(xb, pb, kb >> 5);
    }
#else
    ea = std::exp(xa); eb = std::exp(xb);
#endif
}

// log() for the hot loops (arma prior: log1p(sigma^2/6.25); slice variable: -log1p(-u)), positive normal arguments.
// Table-driven like fast_exp: u = 2^e m, m in [1, 2), j = top 6 mantissa bits, r = m * (1/c_j) - 1 (exact in one FMA,
// |r| <= 1/130), log u = e ln2 + (-log(1/c_j)) + log1p(r) with a degree-7 polynomial: 14 FP64 instructions against ~45
// for libdevice's log1p.  Absolute error <= 2.2e-16 * max(1, |log u|) (CPU emulation against mpmath, and
// tests/test_gpu_parity.py): both uses add the result to O(1) terms.  Anything else (0, denormal, negative, inf, nan)
// goes to libdevice's log.
#if defined(__CUDACC__) || defined(SMCB_DEVMATH)
SMCB_TABLE kLogInvC[64] = {
    0x1.fc07f01fc07f0p-1, 0x1.f44659e4a4271p-1, 0x1.ecc07b301ecc0p-1, 0x1.e573ac901e574p-1,
    0x1.de5d6e3f8868ap-1, 0x1.d77b654b82c34p-1, 0x1.d0cb58f6ec074p-1, 0x1.ca4b3055ee191p-1,
    0x1.c3f8f01c3f8f0p-1, 0x1.bdd2b899406f7p-1, 0x1.b7d6c3dda338bp-1, 0x1.b2036406c80d9p-1,
    0x1.ac5701ac5701bp-1, 0x1.a6d01a6d01a6dp-1, 0x1.a16d3f97a4b02p-1, 0x1.9c2d14ee4a102p-1,
    0x1.970e4f80cb872p-1, 0x1.920fb49d0e229p-1, 0x1.8d3018d3018d3p-1, 0x1.886e5f0abb04ap-1,
    0x1.83c977ab2beddp-1, 0x1.7f405fd017f40p-1, 0x1.7ad2208e0ecc3p-1, 0x1.767dce434a9b1p-1,
    0x1.724287f46debcp-1, 0x1.6e1f76b4337c7p-1, 0x1.6a13cd1537290p-1, 0x1.661ec6a5122f9p-1,
    0x1.623fa77016240p-1, 0x1.5e75bb8d015e7p-1, 0x1.5ac056b015ac0p-1, 0x1.571ed3c506b3ap-1,
    0x1.5390948f40febp-1, 0x1.5015015015015p-1, 0x1.4cab88725af6ep-1, 0x1.49539e3b2d067p-1,
    0x1.460cbc7f5cf9ap-1, 0x1.42d6625d51f87p-1, 0x1.3fb013fb013fbp-1, 0x1.3c995a47babe7p-1,
    0x1.3991c2c187f63p-1, 0x1.3698df3de0748p-1, 0x1.33ae45b57bcb2p-1, 0x1.30d190130d190p-1,
    0x1.2e025c04b8097p-1, 0x1.2b404ad012b40p-1, 0x1.288b01288b013p-1, 0x1.25e22708092f1p-1,
    0x1.23456789abcdfp-1, 0x1.20b470c67c0d9p-1, 0x1.1e2ef3b3fb874p-1, 0x1.1bb4a4046ed29p-1,
    0x1.19453808ca29cp-1, 0x1.16e0689427379p-1, 0x1.1485f0e0acd3bp-1, 0x1.12358e75d3033p-1,
    0x1.0fef010fef011p-1, 0x1.0db20a88f4696p-1, 0x1.0b7e6ec259dc8p-1, 0x1.0953f39010954p-1,
    0x1.073260a47f7c6p-1, 0x1.05197f7d73404p-1, 0x1.03091b51f5e1ap-1, 0x1.0101010101010p-1};
SMCB_TABLE kLogC[64] = {
    0x1.fe02a6b106799p-8, 0x1.7b91b07d5b126p-6, 0x1.39e87b9febd68p-5, 0x1.b42dd711971b9p-5,
    0x1.16536eea37ae3p-4, 0x1.51b073f06183cp-4, 0x1.8c345d6319b23p-4, 0x1.c5e548f5bc743p-4,
    0x1.fec9131dbeabcp-4, 0x1.1b72ad52f67a2p-3, 0x1.371fc201e8f75p-3, 0x1.526e5e3a1b438p-3,
    0x1.6d60fe719d21bp-3, 0x1.87fa06520c911p-3, 0x1.a23bc1fe2b561p-3, 0x1.bc286742d8cd4p-3,
    0x1.d5c216b4fbb94p-3, 0x1.ef0adcbdc5935p-3, 0x1.0402594b4d041p-2, 0x1.1058bf9ae4ad4p-2,
    0x1.1c898c16999fbp-2, 0x1.2895a13de86a4p-2, 0x1.347dd9a987d56p-2, 0x1.404308686a7e4p-2,
    0x1.4be5f957778a1p-2, 0x1.5767717455a6cp-2, 0x1.62c82f2b9c796p-2, 0x1.6e08eaa2ba1e4p-2,
    0x1.792a55fdd47a1p-2, 0x1.842d1da1e8b18p-2, 0x1.8f11e873662c8p-2, 0x1.99d958117e08ap-2,
    0x1.a484090e5bb09p-2, 0x1.af1293247786bp-2, 0x1.b9858969310fdp-2, 0x1.c3dd7a7cdad4dp-2,
    0x1.ce1af0b85f3ecp-2, 0x1.d83e7258a2f3ep-2, 0x1.e24881a7c6c26p-2, 0x1.ec399d2468cc1p-2,
    0x1.f6123fa7028adp-2, 0x1.ffd2e0857f497p-2, 0x1.04bdf9da926d2p-1, 0x1.0986f4f573521p-1,
    0x1.0e44985d1cc8cp-1, 0x1.12f719593efbdp-1, 0x1.179eabbd899a0p-1, 0x1.1c3b81f713c25p-1,
    0x1.20cdcd192ab6ep-1, 0x1.2555bce98f7cap-1, 0x1.29d37fec2b08bp-1, 0x1.2e47436e40268p-1,
    0x1.32b1339121d71p-1, 0x1.37117b54747b6p-1, 0x1.3b68449fffc23p-1, 0x1.3fb5b84d16f43p-1,
    0x1.43f9fe2f9ce67p-1, 0x1.48353d1ea88dfp-1, 0x1.4c679afccee39p-1, 0x1.50913cc01686bp-1,
    0x1.54b2467999498p-1, 0x1.58cadb5cd7989p-1, 0x1.5cdb1dc6c1765p-1, 0x1.60e32f44788d9p-1};
#endif
SMCB_HD double fast_log(double u) {
#if SMCB_TABLE_MATH
    const int hi = dbl_hi(u);
    if (hi < 0x00100000 || hi >= 0x7ff00000) return log(u);
    const int j = (hi >> 14) & 63;
    const double m = dbl_make((hi & 0x000fffff) | 0x3ff00000, dbl_lo(u));
    const double e = (double)((hi >> 20) - 1023);
    const double r = fma(m, SMCB_LDG(&kLogInvC[j]), -1.0);
    double p = fma(1.0 / 7, r, -1.0 / 6);
    p = fma(p, r, 0.2); p = fma(p, r, -0.25); p = fma(p, r, 1.0 / 3); p = fma(p, r, -0.5);
    const double l1 = fma(r * r, p, r);
    return fma(e, 0x1.62e42fefa2000p-1, SMCB_LDG(&kLogC[j])) + fma(e, 0x1.9ef35793c7673p-41, l1);
#else
    return std::log(u);
#endif
}

// log1p of the oracle's statement order (arma prior: log1p(sigma^2/6.25)): glibc log1p on a default host build, the
// table-driven log of 1 + q wherever the table arithmetic is in force (parity device build and its host twin).
SMCB_HD double ref_log1p(double q) {
#if SMCB_TABLE_MATH
    return fast_log(1.0 + q);
#else
    return log1p(q);
#endif
}

// model kinds of the C-ABI (include/smcnuts_b200.h)
enum ModelKind : int { kArma = 0, kPRMwCD = 1, kGauss = 2, kPlugin = 100 };

}  // namespace smcb
