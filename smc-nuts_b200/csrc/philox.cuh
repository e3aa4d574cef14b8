// Philox4x32-10 counter-based streams, one per (seed, iteration, stream-id, particle).
//
// Replaces the reference's single sequential numpy stream shared by all particles
// (/root/reference/smcnuts/proposal/nuts.py:50-53,69,91,99,142; nuts_acc_rej.py:46-47; samples.py:139,155)
// so results are independent of lane scheduling and of the number of GPUs.  The normative CPU
// definition (and the ReplayRNG that serves the same numbers to the unmodified reference) is
// oracle/philox.py; layout:
//   key = (seed lo, seed hi); ctr = (block, iteration<<8 | stream, particle lo, particle hi)
//   draw p -> block p>>1, words (2h, 2h+1), h = p&1;  u = (u64 >> 11) * 2^-53;  Exp(1) = -log1p(-u)
#pragma once
#include "common.cuh"

namespace smcb {

enum Stream : uint32_t {
    kStreamNuts = 0,      // slice variable, directions, merges     (nuts.py:69,91,99,142)
    kStreamMomentum = 1,  // r ~ N(0, I)                            (samples.py:155)
    kStreamAccRej = 2,    // endpoint MH uniform                    (utils.py:32)
    kStreamResample = 3,  // resampling uniforms (particle = slot)  (samples.py:139)
    kStreamInit = 4,      // x0 ~ N(0, I)                           (samples.py:77)
    kStreamEstimate = 5,  // estimate_from_tempered resampling      (estimate_from_tempered.py:43)
    kStreamGQ = 6         // _rng draws of generated quantities     (stan_rng.cuh)
};

struct Philox4 {
    uint32_t w[4];
};

SMCB_HD void mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#if defined(__CUDA_ARCH__)
    lo = a * b;
    hi = __umulhi(a, b);
#else
    uint64_t p = (uint64_t)a * b;
    lo = (uint32_t)p;
    hi = (uint32_t)(p >> 32);
#endif
}

SMCB_HD Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) {
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        uint32_t hi0, lo0, hi1, lo1;
        mulhilo(0xD2511F53u, c0, hi0, lo0);
        mulhilo(0xCD9E8D57u, c2, hi1, lo1);
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    }
    Philox4 o;
    o.w[0] = c0; o.w[1] = c1; o.w[2] = c2; o.w[3] = c3;
    return o;
}

SMCB_HD double u64_to_unit(uint32_t lo, uint32_t hi) {
    uint64_t u = ((uint64_t)hi << 32) | lo;
    return (double)(u >> 11) * 0x1.0p-53;
}

SMCB_HD Philox4 stream_block(uint64_t seed, uint32_t iter, uint32_t stream, uint64_t particle, uint32_t block) {
    return philox4x32_10(block, (iter << 8) | stream, (uint32_t)particle, (uint32_t)(particle >> 32), (uint32_t)seed,
                         (uint32_t)(seed >> 32));
}

// random-access uniform: draw index `draw` of a stream
SMCB_HD double stream_uniform(uint64_t seed, uint32_t iter, uint32_t stream, uint64_t particle, uint32_t draw) {
    Philox4 b = stream_block(seed, iter, stream, particle, draw >> 1);
    return (draw & 1) ? u64_to_unit(b.w[2], b.w[3]) : u64_to_unit(b.w[0], b.w[1]);
}

// Sequential reader of one stream; caches the second half of each Philox block.  The stream identity (seed, iteration and
// stream id, particle) is passed at every draw instead of being stored: in the NUTS kernels it comes from kernel
// arguments (constant bank), and the reader then costs three registers instead of eight.
struct StreamReader {
    uint32_t pos;
    uint32_t c_lo, c_hi;  // cached words 2,3 of the current block

    SMCB_HD void reset() { pos = 0; c_lo = c_hi = 0; }
    // next draw as the 53-bit integer k; the uniform is u = k * 2^-53 (numpy's double construction)
    SMCB_HD uint64_t next_bits(uint64_t seed, uint32_t iter_stream, uint64_t particle) {
        uint64_t k;
        if ((pos & 1) == 0) {
            Philox4 b = philox4x32_10(pos >> 1, iter_stream, (uint32_t)particle, (uint32_t)(particle >> 32),
                                      (uint32_t)seed, (uint32_t)(seed >> 32));
            c_lo = b.w[2]; c_hi = b.w[3];
            k = (((uint64_t)b.w[1] << 32) | b.w[0]) >> 11;
        } else {
            k = (((uint64_t)c_hi << 32) | c_lo) >> 11;
        }
        ++pos;
        return k;
    }
};

// Box-Muller pair j of a stream (draws 2j, 2j+1) -- oracle/philox.py::normals
SMCB_HD void stream_normal_pair(uint64_t seed, uint32_t iter, uint32_t stream, uint64_t particle, uint32_t j,
                                double& z0, double& z1) {
    Philox4 b = stream_block(seed, iter, stream, particle, j);
    double u1 = u64_to_unit(b.w[0], b.w[1]), u2 = u64_to_unit(b.w[2], b.w[3]);
    double rad = sqrt(-2.0 * log1p(-u1));
    double ang = kTwoPi * u2;
    z0 = rad * cos(ang);
    z1 = rad * sin(ang);
}

}  // namespace smcb
