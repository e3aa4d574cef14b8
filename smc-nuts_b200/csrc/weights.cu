// K4, K5, K7, K8, K12 -- HBM-bound per-particle kernels: Philox fills, weight updates, online
// log-sum-exp / ESS, the multi-candidate tempering objective, weighted moments.
//
// All are grid-stride over particles with the grid a multiple of the SM count; reductions finish in a
// single launch ("last block reduces the per-block partials in a fixed order" -> deterministic).
#include "bisect.cuh"
#include "capi.cuh"
#include "philox.cuh"

namespace smcb {

constexpr int kRedThreads = 256;
constexpr int kRedMaxBlocks = 2048;
constexpr int kRedMaxVals = 256;  // doubles of partial state per block
constexpr long long kRedWsBytes = (long long)kRedMaxBlocks * kRedMaxVals * 8 + 256;

__device__ __forceinline__ double map_lp(double lp) { return is_finite(lp) ? lp : neg_inf(); }

// ------------------------------------------------------------------------------------------ Philox fills
__global__ void normals_kernel(uint64_t seed, uint32_t iter, uint32_t stream, uint64_t p0, long long N, int D,
                               double* __restrict__ out) {
    const int npair = (D + 1) / 2;
    const long long total = N * npair;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const long long i = t / npair;
        const int j = (int)(t - i * npair);
        double z0, z1;
        stream_normal_pair(seed, iter, stream, p0 + (uint64_t)i, (uint32_t)j, z0, z1);
        out[i * D + 2 * j] = z0;
        if (2 * j + 1 < D) out[i * D + 2 * j + 1] = z1;
    }
}

__global__ void uniforms_kernel(uint64_t seed, uint32_t iter, uint32_t stream, uint64_t p0, long long N, uint32_t draw,
                                double* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x)
        out[i] = stream_uniform(seed, iter, stream, p0 + (uint64_t)i, draw);
}

// ------------------------------------------------------------------------------------------ row norms
// 0.5*|row|^2 for row-major [N, D]: coalesced flat loads into smem, then one thread per row.
template <int ROWS>
__device__ __forceinline__ void tile_half_sqnorm(const double* __restrict__ r, long long row0, long long N, int D,
                                                 double* sm, double* out_local) {
    const long long e0 = row0 * D;
    const long long ne = min((long long)ROWS, N - row0) * D;
    for (long long e = threadIdx.x; e < ne; e += blockDim.x) sm[e + e / D] = r[e0 + e];  // +1 pad per row
    __syncthreads();
    if (threadIdx.x < ROWS && row0 + threadIdx.x < N) {
        const double* rowp = sm + (size_t)threadIdx.x * (D + 1);
        double s = 0.0;
        for (int d = 0; d < D; ++d) s += rowp[d] * rowp[d];
        *out_local = 0.5 * s;
    }
    __syncthreads();
}

// Cooperative variant for D = 2*LPR (LPR = lanes per row, a power of two): LPR adjacent lanes read one row as
// 16-byte chunks, so every warp-level load covers 32/LPR whole rows = 512 contiguous bytes; the squares are folded
// with log2(LPR) shuffles.  ROWS_PER_ITER rows per group are in flight to keep enough bytes outstanding.
// The groups of one warp can run different trip counts of their row loops, so a shuffle names only its own group's
// lanes (every xor offset is < LPR: the exchange never leaves the group).
template <int LPR>
__device__ __forceinline__ unsigned group_mask() {
    return LPR == 32 ? 0xffffffffu : ((1u << (LPR & 31)) - 1u) << ((threadIdx.x & 31) & ~(LPR - 1));
}
template <int LPR>
__device__ __forceinline__ double group_half_sqnorm(const double* __restrict__ rowp, int sub) {
    const double2 v = *reinterpret_cast<const double2*>(rowp + 2 * sub);
    double s = v.x * v.x + v.y * v.y;
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) s += __shfl_xor_sync(group_mask<LPR>(), s, o);
    return 0.5 * s;
}

template <int LPR>
__global__ void __launch_bounds__(256) reweight_forward_coop_kernel(const double* __restrict__ logw,
                                                                    const double* __restrict__ lp_x,
                                                                    const double* __restrict__ lp_xnew,
                                                                    const double* __restrict__ r,
                                                                    const double* __restrict__ r_new, long long N,
                                                                    double* __restrict__ out) {
    constexpr int D = 2 * LPR, U = LPR < 4 ? LPR : 4;  // lane `sub` < U of a group finishes row i0 + sub
    const int sub = threadIdx.x % LPR;
    const long long group = (blockIdx.x * (long long)blockDim.x + threadIdx.x) / LPR;
    const long long ngroups = (long long)gridDim.x * blockDim.x / LPR;
    const long long nfull = (N / U) * U;
    for (long long i0 = group * U; i0 < nfull; i0 += ngroups * U) {
        double2 a[U], b[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            a[u] = *reinterpret_cast<const double2*>(r + (i0 + u) * D + 2 * sub);
            b[u] = *reinterpret_cast<const double2*>(r_new + (i0 + u) * D + 2 * sub);
        }
        double k0[U], k1[U];
#pragma unroll
        for (int u = 0; u < U; ++u) { k0[u] = a[u].x * a[u].x + a[u].y * a[u].y; k1[u] = b[u].x * b[u].x + b[u].y * b[u].y; }
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1)
#pragma unroll
            for (int u = 0; u < U; ++u) {
                k0[u] += __shfl_xor_sync(group_mask<LPR>(), k0[u], o);
                k1[u] += __shfl_xor_sync(group_mask<LPR>(), k1[u], o);
            }
        if (sub < U) {  // lane `sub` of the group finishes row i0 + sub: coalesced 8-byte scalars
            double kk0 = k0[0], kk1 = k1[0];
#pragma unroll
            for (int u = 1; u < U; ++u) if (sub == u) { kk0 = k0[u]; kk1 = k1[u]; }
            const long long i = i0 + sub;
            out[i] = logw[i] + lp_xnew[i] - lp_x[i] + (-0.5 * kk1) - (-0.5 * kk0);
        }
    }
    // tail rows (N % U)
    for (long long i = nfull + group; i < N; i += ngroups) {
        const double k0 = group_half_sqnorm<LPR>(r + i * D, sub), k1 = group_half_sqnorm<LPR>(r_new + i * D, sub);
        if (sub == 0) out[i] = logw[i] + lp_xnew[i] - lp_x[i] + (-k1) - (-k0);
    }
}

__global__ void row_half_sqnorm_kernel(const double* __restrict__ r, long long N, int D, double* __restrict__ out) {
    extern __shared__ double sm[];
    constexpr int ROWS = kRedThreads;
    for (long long row0 = (long long)blockIdx.x * ROWS; row0 < N; row0 += (long long)gridDim.x * ROWS) {
        double v = 0.0;
        tile_half_sqnorm<ROWS>(r, row0, N, D, sm, &v);
        if (row0 + threadIdx.x < N) out[row0 + threadIdx.x] = v;
    }
}

__global__ void std_normal_logpdf_kernel(const double* __restrict__ x, long long N, int D, double* __restrict__ out) {
    extern __shared__ double sm[];
    constexpr int ROWS = kRedThreads;
    for (long long row0 = (long long)blockIdx.x * ROWS; row0 < N; row0 += (long long)gridDim.x * ROWS) {
        double v = 0.0;
        tile_half_sqnorm<ROWS>(x, row0, N, D, sm, &v);
        if (row0 + threadIdx.x < N) out[row0 + threadIdx.x] = -v - 0.5 * D * kLog2Pi;
    }
}

// Rows too wide for the shared-memory tile (D > 110): one warp per row, lanes stride over the coordinates.
// mode 0: out = 0.5|row|^2;  1: out = -0.5|row|^2 - D/2 log 2pi;  2: out = aux - (-0.5|row|^2 - D/2 log 2pi)
__global__ void __launch_bounds__(256) row_sqnorm_warp_kernel(const double* __restrict__ r, long long N, int D, int mode,
                                                               const double* __restrict__ aux, double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long i = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < N; i += nwarps) {
        double s = 0.0;
        for (int d = lane; d < D; d += 32) { const double v = r[i * D + d]; s += v * v; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
            const double h = 0.5 * s, lg = -h - 0.5 * D * kLog2Pi;
            out[i] = mode == 0 ? h : mode == 1 ? lg : aux[i] - lg;
        }
    }
}
__global__ void __launch_bounds__(256) reweight_forward_warp_kernel(const double* __restrict__ logw,
                                                                     const double* __restrict__ lp_x,
                                                                     const double* __restrict__ lp_xnew,
                                                                     const double* __restrict__ r,
                                                                     const double* __restrict__ r_new, long long N, int D,
                                                                     double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    const double c = 0.5 * D * kLog2Pi;
    for (long long i = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < N; i += nwarps) {
        double s0 = 0.0, s1 = 0.0;
        for (int d = lane; d < D; d += 32) {
            const double a = r[i * D + d], b = r_new[i * D + d];
            s0 += a * a; s1 += b * b;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); }
        if (lane == 0) out[i] = logw[i] + lp_xnew[i] - lp_x[i] + (-0.5 * s1 - c) - (-0.5 * s0 - c);
    }
}

__global__ void uniform_logw_kernel(const double* __restrict__ logZ, double logN, long long N, double* __restrict__ out) {
    const double v = logZ[0] - logN;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) out[i] = v;
}

__global__ void affine_kernel(const double* __restrict__ in, long long N, double a, double b, double* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x)
        out[i] = a * in[i] + b;
}

__global__ void init_logw_kernel(const double* __restrict__ lp, const double* __restrict__ x, long long N, int D,
                                 double* __restrict__ logw) {
    extern __shared__ double sm[];
    constexpr int ROWS = kRedThreads;
    for (long long row0 = (long long)blockIdx.x * ROWS; row0 < N; row0 += (long long)gridDim.x * ROWS) {
        double v = 0.0;
        tile_half_sqnorm<ROWS>(x, row0, N, D, sm, &v);
        const long long i = row0 + threadIdx.x;
        if (i < N) logw[i] = lp[i] - (-v - 0.5 * D * kLog2Pi);
    }
}

__global__ void reweight_forward_kernel(const double* __restrict__ logw, const double* __restrict__ lp_x,
                                        const double* __restrict__ lp_xnew, const double* __restrict__ r,
                                        const double* __restrict__ r_new, long long N, int D,
                                        double* __restrict__ out) {
    extern __shared__ double sm[];
    constexpr int ROWS = kRedThreads;
    const double c = 0.5 * D * kLog2Pi;
    for (long long row0 = (long long)blockIdx.x * ROWS; row0 < N; row0 += (long long)gridDim.x * ROWS) {
        double k0 = 0.0, k1 = 0.0;
        tile_half_sqnorm<ROWS>(r, row0, N, D, sm, &k0);
        tile_half_sqnorm<ROWS>(r_new, row0, N, D, sm, &k1);
        const long long i = row0 + threadIdx.x;
        if (i < N) out[i] = logw[i] + lp_xnew[i] - lp_x[i] + (-k1 - c) - (-k0 - c);
    }
}

__global__ void reweight_forward_ke_kernel(const double* __restrict__ logw, const double* __restrict__ lp_x,
                                           const double* __restrict__ lp_xnew, const double* __restrict__ ke_old,
                                           const double* __restrict__ ke_new, long long N, double* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x)
        out[i] = logw[i] + lp_xnew[i] - lp_x[i] + (-ke_new[i]) - (-ke_old[i]);
}

// the same with logp(x) and logp(x_new) formed in place from the split densities the NUTS kernel emitted
// (A + phi*B, non-finite -> -inf as smcb_combine_logp): one launch instead of three per SMC iteration
__global__ void reweight_forward_split_kernel(const double* __restrict__ logw, const double* __restrict__ A_old,
                                              const double* __restrict__ B_old, const double* __restrict__ A_new,
                                              const double* __restrict__ B_new, const double* __restrict__ ke_old,
                                              const double* __restrict__ ke_new, double phi, long long N,
                                              double* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
        const double lp_x = map_lp(A_old[i] + phi * B_old[i]), lp_xnew = map_lp(A_new[i] + phi * B_new[i]);
        out[i] = logw[i] + lp_xnew - lp_x + (-ke_new[i]) - (-ke_old[i]);
    }
}

__global__ void reweight_general_kernel(const double* __restrict__ logw, const double* __restrict__ lp_x,
                                        const double* __restrict__ lp_xnew, const double* __restrict__ L,
                                        const double* __restrict__ q, long long N, double* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x)
        out[i] = logw[i] + lp_xnew[i] - lp_x[i] + L[i] - q[i];
}

__global__ void reweight_asymptotic_kernel(const double* __restrict__ logw, const double* __restrict__ A,
                                           const double* __restrict__ B, double phi_new, double phi_old, long long N,
                                           double* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x)
        out[i] = logw[i] + map_lp(A[i] + phi_new * B[i]) - map_lp(A[i] + phi_old * B[i]);
}

__global__ void tempering_arrays_kernel(const double* __restrict__ A, const double* __restrict__ B, double phi_old,
                                        long long N, double* __restrict__ logpri, double* __restrict__ loglik,
                                        double* __restrict__ c) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
        const double a = A[i], b = B[i];
        const double pri = map_lp(a + 0.0 * b);
        logpri[i] = pri;
        loglik[i] = map_lp(a + b) - pri;
        c[i] = map_lp(a + phi_old * b);
    }
}

// ------------------------------------------------------------------------------------------ online LSE
struct Lse {
    double m, s1, s2;
};
__device__ __forceinline__ Lse lse_empty() { return Lse{neg_inf(), 0.0, 0.0}; }
__device__ __forceinline__ void lse_push(Lse& a, double x) {
    if (x == neg_inf()) return;  // samples.py:96 / adaptive_tempering.py:46: -inf entries are dropped
    if (x > a.m) {
        const double f = fast_exp(a.m - x);  // exp(-inf) = 0 on the first element
        a.s1 = a.s1 * f + 1.0;
        a.s2 = a.s2 * f * f + 1.0;
        a.m = x;
    } else {
        const double e = fast_exp(x - a.m);  // NaN input poisons the sums, as in scipy.logsumexp
        a.s1 += e;
        a.s2 += e * e;
    }
}
__device__ __forceinline__ Lse lse_merge(const Lse& a, const Lse& b) {
    if (b.s1 == 0.0 && b.m == neg_inf()) return a;
    if (a.s1 == 0.0 && a.m == neg_inf()) return b;
    Lse o;
    o.m = (a.m > b.m) ? a.m : b.m;
    if (a.m != a.m || b.m != b.m) o.m = a.m + b.m;  // NaN
    const double fa = exp(a.m - o.m), fb = exp(b.m - o.m);
    o.s1 = a.s1 * fa + b.s1 * fb;
    o.s2 = a.s2 * fa * fa + b.s2 * fb * fb;
    return o;
}
__device__ __forceinline__ Lse lse_warp_reduce(Lse v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Lse w;
        w.m = __shfl_xor_sync(0xffffffffu, v.m, o);
        w.s1 = __shfl_xor_sync(0xffffffffu, v.s1, o);
        w.s2 = __shfl_xor_sync(0xffffffffu, v.s2, o);
        // fixed combination order (lower lane first) keeps the result identical on both partners
        v = ((threadIdx.x & 31) & o) ? lse_merge(w, v) : lse_merge(v, w);
    }
    return v;
}

// Block-level reduce of NV Lse states per thread, then "last block" merges all block partials in block order.
// partial layout: ws[block][NV*3]; counter at ws + kRedMaxBlocks*kRedMaxVals.
template <int NV>
__device__ void lse_block_finish(Lse (&v)[NV], double* ws, double* out, int nv) {
    __shared__ double sh[(kRedThreads / 32) * NV * 3];
    __shared__ bool is_last;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        Lse r = lse_warp_reduce(v[j]);
        if (lane == 0) { sh[(warp * NV + j) * 3] = r.m; sh[(warp * NV + j) * 3 + 1] = r.s1; sh[(warp * NV + j) * 3 + 2] = r.s2; }
    }
    __syncthreads();
    if (threadIdx.x < nv) {
        const int j = threadIdx.x;
        Lse r = lse_empty();
        for (int w = 0; w < kRedThreads / 32; ++w)
            r = lse_merge(r, Lse{sh[(w * NV + j) * 3], sh[(w * NV + j) * 3 + 1], sh[(w * NV + j) * 3 + 2]});
        double* p = ws + (size_t)blockIdx.x * kRedMaxVals + j * 3;
        p[0] = r.m; p[1] = r.s1; p[2] = r.s2;
    }
    __threadfence();
    __syncthreads();
    unsigned* counter = (unsigned*)(ws + (size_t)kRedMaxBlocks * kRedMaxVals);
    if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (is_last) {  // all threads of the last block merge the per-block partials: strided, then warp/block tree
        __threadfence();
        for (int j = 0; j < nv; ++j) {
            Lse r = lse_empty();
            for (unsigned b = threadIdx.x; b < gridDim.x; b += kRedThreads) {
                const volatile double* p = ws + (size_t)b * kRedMaxVals + j * 3;
                r = lse_merge(r, Lse{p[0], p[1], p[2]});
            }
            r = lse_warp_reduce(r);
            __syncthreads();
            if (lane == 0) { sh[warp * 3] = r.m; sh[warp * 3 + 1] = r.s1; sh[warp * 3 + 2] = r.s2; }
            __syncthreads();
            if (threadIdx.x == 0) {
                Lse t = lse_empty();
                for (int w = 0; w < kRedThreads / 32; ++w) t = lse_merge(t, Lse{sh[w * 3], sh[w * 3 + 1], sh[w * 3 + 2]});
                out[j * 3] = t.m; out[j * 3 + 1] = t.s1; out[j * 3 + 2] = t.s2;
            }
        }
        if (threadIdx.x == 0) *counter = 0;
    }
}

// Four elements at once: one running-max update (rare after the first few elements), then four independent exps --
// no per-element branch on the running maximum, 16-byte loads.  Same semantics as lse_push element by element
// (-inf dropped, NaN poisons, an element equal to the maximum counts exactly 1).
__device__ __forceinline__ void lse_push4(Lse& a, double x0, double x1, double x2, double x3) {
    double mn = a.m;
    mn = (x0 > mn) ? x0 : mn; mn = (x1 > mn) ? x1 : mn; mn = (x2 > mn) ? x2 : mn; mn = (x3 > mn) ? x3 : mn;
    if (mn > a.m) {
        const double f = fast_exp(a.m - mn);   // exp(-inf) = 0 on the first finite element
        a.s1 *= f; a.s2 *= f * f; a.m = mn;
    }
    const double ninf = neg_inf();
    double e0, e1, e2, e3;
    fast_exp_pair(x0 - mn, x1 - mn, e0, e1);
    fast_exp_pair(x2 - mn, x3 - mn, e2, e3);
    e0 = (x0 == mn) ? 1.0 : e0; e1 = (x1 == mn) ? 1.0 : e1; e2 = (x2 == mn) ? 1.0 : e2; e3 = (x3 == mn) ? 1.0 : e3;
    e0 = (x0 == ninf) ? 0.0 : e0; e1 = (x1 == ninf) ? 0.0 : e1; e2 = (x2 == ninf) ? 0.0 : e2; e3 = (x3 == ninf) ? 0.0 : e3;
    a.s1 += (e0 + e1) + (e2 + e3);
    a.s2 += (e0 * e0 + e1 * e1) + (e2 * e2 + e3 * e3);
}

__global__ void __launch_bounds__(kRedThreads) lse_partial_kernel(const double* __restrict__ logw, long long N,
                                                                   double* out3, double* ws) {
    Lse v[1] = {lse_empty()};
    const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x, nthr = (long long)gridDim.x * blockDim.x;
    if ((reinterpret_cast<uintptr_t>(logw) & 15) == 0) {
        // Software-pipelined: the loads of the next pair of quads are issued before the exps of the current pair, so the
        // DRAM latency of a round hides behind ~300 issue cycles of arithmetic per warp instead of adding to them
        // (ncu, round 2: 108 us for 2^25 elements with the loads consumed right after they were issued).
        const long long nq = N / 4;
        const double2* p = reinterpret_cast<const double2*>(logw);
        const double ninf = neg_inf();
        const double2 pad = make_double2(ninf, ninf);   // a missing quad contributes nothing
        long long q = tid;
        double2 a0 = pad, b0 = pad, a1 = pad, b1 = pad;
        if (q < nq) { a0 = p[2 * q]; b0 = p[2 * q + 1]; }
        if (q + nthr < nq) { a1 = p[2 * (q + nthr)]; b1 = p[2 * (q + nthr) + 1]; }
        while (q < nq) {
            const long long qn = q + 2 * nthr;
            double2 na0 = pad, nb0 = pad, na1 = pad, nb1 = pad;
            if (qn < nq) { na0 = p[2 * qn]; nb0 = p[2 * qn + 1]; }
            if (qn + nthr < nq) { na1 = p[2 * (qn + nthr)]; nb1 = p[2 * (qn + nthr) + 1]; }
            lse_push4(v[0], a0.x, a0.y, b0.x, b0.y);
            if (q + nthr < nq) lse_push4(v[0], a1.x, a1.y, b1.x, b1.y);
            a0 = na0; b0 = nb0; a1 = na1; b1 = nb1;
            q = qn;
        }
        for (long long i = 4 * nq + tid; i < N; i += nthr) lse_push(v[0], logw[i]);
    } else {
        for (long long i = tid; i < N; i += nthr) lse_push(v[0], logw[i]);
    }
    lse_block_finish<1>(v, ws, out3, 1);
}

__global__ void lse_finalize_kernel(const double* __restrict__ triples, int P, double* __restrict__ out2) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        Lse r = lse_empty();
        for (int p = 0; p < P; ++p) r = lse_merge(r, Lse{triples[3 * p], triples[3 * p + 1], triples[3 * p + 2]});
        out2[0] = r.m + log(r.s1);          // logsumexp  (samples.py:98)
        out2[1] = (r.s1 * r.s1) / r.s2;     // 1 / sum(wn^2) (samples.py:113)
    }
}

__global__ void normalise_kernel(const double* __restrict__ logw, long long N, const double* __restrict__ logZ,
                                 double* __restrict__ wn) {
    const double z = *logZ;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
        const double x = logw[i];
        wn[i] = (x == neg_inf()) ? 0.0 : fast_exp(x - z);
    }
}

constexpr int kMaxPhi = 16;
template <int NV>
__global__ void __launch_bounds__(kRedThreads) ess_multi_phi_kernel(const double* __restrict__ loglik,
                                                                     const double* __restrict__ logpri,
                                                                     const double* __restrict__ c, long long N,
                                                                     const double* __restrict__ phis, int m,
                                                                     double* out, double* ws) {
    Lse v[NV];
    double ph[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) { v[j] = lse_empty(); ph[j] = (j < m) ? phis[j] : 0.0; }
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
        const double ll = loglik[i], pri = logpri[i], cc = c[i];
#pragma unroll
        for (int j = 0; j < NV; ++j)
            if (j < m) lse_push(v[j], (ph[j] * ll + pri) - cc);  // adaptive_tempering.py:43 (same association as numpy)
    }
    lse_block_finish<NV>(v, ws, out, m);
}

// ---- device-resident bisection (bisect.cuh): candidates come from, and results go back into, a BisectState in
//      device memory; every kernel is a no-op once the state has left kBisectRunning, so the host can enqueue the
//      whole fixed schedule of passes without looking at intermediate results.
__global__ void bisect_init_kernel(BisectState* s, double xa, double xb, double target) {
    if (threadIdx.x == 0 && blockIdx.x == 0)
        bisect_init(*s, xa, xb, target, 2e-12, 8.881784197001252e-16, 100);   // scipy.optimize.bisect defaults
}

// objective pass straight from the split log density: logpri = A, loglik = (A + B) - A, c = A + phi_old B with the
// -inf failure mapping (adaptive_tempering.py:38-43, samples.py:207) formed on the fly -- 16 bytes read per particle,
// nothing written.  out[kBisectMaxCand][3] (unused candidates: empty states).
__global__ void __launch_bounds__(kRedThreads) bisect_eval_kernel(const double* __restrict__ A,
                                                                   const double* __restrict__ B, double phi_old,
                                                                   long long N, const BisectState* s, double* out,
                                                                   double* ws) {
    if (s->status != kBisectRunning) return;
    constexpr int NV = kBisectMaxCand;
    const int m = s->n_cand;
    Lse v[NV];
    double ph[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) { v[j] = lse_empty(); ph[j] = (j < m) ? s->cand[j] : 0.0; }
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
        const double a = A[i], b = B[i];
        const double pri = map_lp(a + 0.0 * b);
        const double ll = map_lp(a + b) - pri;
        const double cc = map_lp(a + phi_old * b);
#pragma unroll
        for (int j = 0; j < NV; ++j)
            if (j < m) lse_push(v[j], (ph[j] * ll + pri) - cc);
    }
    lse_block_finish<NV>(v, ws, out, NV);
}

// merge the P rank states of every candidate (rank order), f = ESS - target, walk the tree, prepare the next pass
__global__ void bisect_step_kernel(const double* __restrict__ triples, int P, BisectState* s) {
    __shared__ double f[kBisectMaxCand];
    if (s->status != kBisectRunning) return;
    const int j = threadIdx.x;
    if (j < kBisectMaxCand) {
        Lse r = lse_empty();
        for (int p = 0; p < P; ++p) {
            const double* t = triples + ((size_t)p * kBisectMaxCand + j) * 3;
            r = lse_merge(r, Lse{t[0], t[1], t[2]});
        }
        f[j] = (r.s1 * r.s1) / r.s2 - s->target;     // adaptive_tempering.py:54-56
    }
    __syncthreads();
    if (j == 0) bisect_advance(*s, f);
}

__global__ void bisect_read_kernel(const BisectState* s, double* out4) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        out4[0] = s->result; out4[1] = (double)s->status; out4[2] = (double)s->iterations; out4[3] = s->nan_at;
    }
}

// ------------------------------------------------------------------------------------------ weighted moments
// out[d] = sum_i wn_i * (c(x_i)_d - center_d)^power.  Thread t owns column (t % D) of a flat coalesced sweep whose
// stride is a multiple of D.
__global__ void __launch_bounds__(kRedThreads) weighted_moment_kernel(const double* __restrict__ x,
                                                                       const double* __restrict__ wn, long long N,
                                                                       int D, int constrain,
                                                                       const double* __restrict__ center, int power,
                                                                       double* out, double* ws, int threads_used) {
    __shared__ double sh[kRedThreads];
    __shared__ bool is_last;
    const long long total = N * D;
    const long long gstride = (long long)gridDim.x * threads_used;
    double acc = 0.0;
    const int col = threadIdx.x % D;
    if ((int)threadIdx.x < threads_used) {
        const double cen = center ? center[col] : 0.0;
        const bool do_exp = (constrain == SMCB_CONSTRAIN_EXP_LAST) && (col == D - 1);
        // the sweep stride is a multiple of D, so the row index advances by a constant: no 64-bit division per element
        long long row = (long long)blockIdx.x * (threads_used / D) + (int)threadIdx.x / D;
        const long long rstride = gstride / D;
        for (long long e = (long long)blockIdx.x * threads_used + threadIdx.x; e < total; e += gstride, row += rstride) {
            double v = x[e];
            if (do_exp) v = fast_exp(v);
            v -= cen;
            if (power == 2) v *= v;
            acc += wn[row] * v;
        }
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    if ((int)threadIdx.x < D) {
        double s = 0.0;
        for (int t = threadIdx.x; t < threads_used; t += D) s += sh[t];
        ws[(size_t)blockIdx.x * kRedMaxVals + threadIdx.x] = s;
    }
    __threadfence();
    __syncthreads();
    unsigned* counter = (unsigned*)(ws + (size_t)kRedMaxBlocks * kRedMaxVals);
    if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (is_last) {  // thread t sums column (t % D) over blocks t/D, t/D + used/D, ...; then the same column fold
        __threadfence();
        double a2 = 0.0;
        if ((int)threadIdx.x < threads_used)
            for (unsigned b = threadIdx.x / D; b < gridDim.x; b += threads_used / D)
                a2 += ((const volatile double*)ws)[(size_t)b * kRedMaxVals + col];
        __syncthreads();
        sh[threadIdx.x] = a2;
        __syncthreads();
        if ((int)threadIdx.x < D) {
            double s = 0.0;
            for (int t = threadIdx.x; t < threads_used; t += D) s += sh[t];
            out[threadIdx.x] = s;
        }
        if (threadIdx.x == 0) *counter = 0;
    }
}

// One pass for both moments about a caller-supplied centre c (the previous iteration's mean: close to this one's, so
// the second central moment m2 - m1^2 loses nothing to cancellation):
//   out[d] = sum_i wn_i (c(x_i)_d - c_d),  out[D + d] = sum_i wn_i (c(x_i)_d - c_d)^2.
// Reads x and wn once instead of twice, and a sharded run all-reduces the 2D sums in ONE collective instead of two
// (estimate.py:91-93 computes the mean first and then the variance about it).  Same thread mapping as above.
__global__ void __launch_bounds__(kRedThreads) weighted_moments12_kernel(const double* __restrict__ x,
                                                                          const double* __restrict__ wn, long long N,
                                                                          int D, int constrain,
                                                                          const double* __restrict__ center, double* out,
                                                                          double* ws, int threads_used) {
    __shared__ double sh[2 * kRedThreads];
    __shared__ bool is_last;
    const long long total = N * D;
    const long long gstride = (long long)gridDim.x * threads_used;
    double a1 = 0.0, a2 = 0.0;
    const int col = threadIdx.x % D;
    if ((int)threadIdx.x < threads_used) {
        const double cen = center ? center[col] : 0.0;
        const bool do_exp = (constrain == SMCB_CONSTRAIN_EXP_LAST) && (col == D - 1);
        long long row = (long long)blockIdx.x * (threads_used / D) + (int)threadIdx.x / D;
        const long long rstride = gstride / D;
        for (long long e = (long long)blockIdx.x * threads_used + threadIdx.x; e < total; e += gstride, row += rstride) {
            double v = x[e];
            if (do_exp) v = fast_exp(v);
            v -= cen;
            const double w = wn[row];
            a1 += w * v;
            a2 += w * (v * v);
        }
    }
    sh[threadIdx.x] = a1; sh[kRedThreads + threadIdx.x] = a2;
    __syncthreads();
    if ((int)threadIdx.x < 2 * D) {
        const int c = threadIdx.x % D, which = threadIdx.x / D;
        double s = 0.0;
        for (int t = c; t < threads_used; t += D) s += sh[which * kRedThreads + t];
        ws[(size_t)blockIdx.x * kRedMaxVals + threadIdx.x] = s;
    }
    __threadfence();
    __syncthreads();
    unsigned* counter = (unsigned*)(ws + (size_t)kRedMaxBlocks * kRedMaxVals);
    if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (is_last) {
        __threadfence();
        double b1 = 0.0, b2 = 0.0;
        if ((int)threadIdx.x < threads_used)
            for (unsigned b = threadIdx.x / D; b < gridDim.x; b += threads_used / D) {
                b1 += ((const volatile double*)ws)[(size_t)b * kRedMaxVals + col];
                b2 += ((const volatile double*)ws)[(size_t)b * kRedMaxVals + D + col];
            }
        __syncthreads();
        sh[threadIdx.x] = b1; sh[kRedThreads + threadIdx.x] = b2;
        __syncthreads();
        if ((int)threadIdx.x < 2 * D) {
            const int c = threadIdx.x % D, which = threadIdx.x / D;
            double s = 0.0;
            for (int t = c; t < threads_used; t += D) s += sh[which * kRedThreads + t];
            out[threadIdx.x] = s;
        }
        if (threadIdx.x == 0) *counter = 0;
    }
}

// mean = c + m1, var = m2 - m1^2 from the (all-reduced) sums of the kernel above
__global__ void moments12_finalize_kernel(const double* __restrict__ sums, const double* __restrict__ center, int D,
                                          double* __restrict__ mean, double* __restrict__ var) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d < D) {
        const double m1 = sums[d], m2 = sums[D + d];
        mean[d] = (center ? center[d] : 0.0) + m1;
        const double v = m2 - m1 * m1;
        var[d] = (v < 0.0) ? 0.0 : v;   // a sum of non-negative terms in the two-pass form: never negative there (NaN passes)
    }
}

__global__ void __launch_bounds__(kRedThreads) count_moved_kernel(const double* __restrict__ x,
                                                                   const double* __restrict__ xn, long long N, int D,
                                                                   double* out, double* ws) {
    __shared__ double sh[kRedThreads / 32];
    __shared__ bool is_last;
    double cnt = 0.0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
        bool all = true;
        for (int d = 0; d < D; ++d) all = all && (x[i * D + d] != xn[i * D + d]);
        cnt += all ? 1.0 : 0.0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < kRedThreads / 32; ++w) s += sh[w];
        ws[(size_t)blockIdx.x * kRedMaxVals] = s;
    }
    __threadfence();
    __syncthreads();
    unsigned* counter = (unsigned*)(ws + (size_t)kRedMaxBlocks * kRedMaxVals);
    if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (is_last) {
        __threadfence();
        double s = 0.0;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += kRedThreads) s += ((const volatile double*)ws)[(size_t)b * kRedMaxVals];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < kRedThreads / 32; ++w) t += sh[w];
            out[0] = t;
            *counter = 0;
        }
    }
}

// sum of an array in a wider accumulator: int32 -> int64 (the grad-eval counter of the metric), double -> double (the
// acceptance statistic of the step-size adaptation); fixed tile order, so the result does not depend on scheduling
template <typename T, typename Acc>
__global__ void __launch_bounds__(kRedThreads) sum_kernel(const T* __restrict__ v, long long N, Acc* out, double* ws) {
    static_assert(sizeof(Acc) == sizeof(double), "partials share the reduction workspace");
    __shared__ Acc sh[kRedThreads / 32];
    __shared__ bool is_last;
    Acc acc = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) acc += v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    Acc* wsl = (Acc*)ws;
    if (threadIdx.x == 0) {
        Acc s = 0;
        for (int w = 0; w < kRedThreads / 32; ++w) s += sh[w];
        wsl[(size_t)blockIdx.x * kRedMaxVals] = s;
    }
    __threadfence();
    __syncthreads();
    unsigned* counter = (unsigned*)(ws + (size_t)kRedMaxBlocks * kRedMaxVals);
    if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (is_last) {
        __threadfence();
        Acc s = 0;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += kRedThreads) s += ((const volatile Acc*)wsl)[(size_t)b * kRedMaxVals];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            Acc t = 0;
            for (int w = 0; w < kRedThreads / 32; ++w) t += sh[w];
            out[0] = t;
            *counter = 0;
        }
    }
}

// out[i][d] = x[i][d] * scale[d] (inverse = 0) or x[i][d] / scale[d] (inverse = 1): the change of variables of the
// diagonal-metric NUTS path (ScaledModel, models.cuh) at the kernel's boundaries
__global__ void scale_rows_kernel(const double* __restrict__ x, long long n_elem, int D, const double* __restrict__ scale,
                                  int inverse, double* __restrict__ out) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_elem; e += (long long)gridDim.x * blockDim.x) {
        const double s = scale[(int)(e % D)];
        out[e] = inverse ? x[e] / s : x[e] * s;
    }
}

// out[i][d] = accepted[i] ? z[i][d] * scale[d] : x[i][d]: back to x-space after a diagonal-metric transition with the MH
// epilogue, where a rejected particle must keep its x row (the kernel returned z = x / scale for it, and z * scale need not
// round back to x).  out may alias z.
__global__ void scale_rows_accepted_kernel(const double* z, const int* __restrict__ accepted, const double* __restrict__ x,
                                           long long n_elem, int D, const double* __restrict__ scale, double* out) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_elem; e += (long long)gridDim.x * blockDim.x) {
        const int d = (int)(e % D);
        out[e] = accepted[e / D] ? z[e] * scale[d] : x[e];
    }
}

// ------------------------------------------------------------------------------------------ FP64 probe
__global__ void probe_fp64_kernel(int iters, double* sink) {
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-7;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.678) sink[0] = s;  // never true; keeps the loop alive
}

__global__ void fast_log_kernel(const double* __restrict__ x, long long N, double* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x)
        out[i] = fast_log(x[i]);
}

__global__ void fast_exp_kernel(const double* __restrict__ x, long long N, double* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x)
        out[i] = fast_exp(x[i]);
}

// FP64 tensor-core probe: 8 independent mma.m8n8k4 accumulator chains per warp
__global__ void probe_dmma_kernel(int iters, double* sink) {
    double c[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) c[i] = threadIdx.x * 1e-9 + i;
    const double a = 1.0000001, b = 0.9999999;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                         : "+d"(c[2 * j]), "+d"(c[2 * j + 1]) : "d"(a), "d"(b));
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += c[i];
    if (s == 12345.678) sink[0] = s;
}

// One mma.m8n8k4 per warp on caller-supplied fragments (a[32], b[32], c[64] -> out[64]; lane l holds a[l], b[l],
// c[2l], c[2l+1]): lets a test establish the rounding / association of the FP64 tensor-core instruction against an
// exact CPU model.
__global__ void debug_dmma_kernel(const double* __restrict__ a, const double* __restrict__ b,
                                  const double* __restrict__ c, double* __restrict__ out, int nwarps) {
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), l = threadIdx.x & 31;
    if (w >= nwarps) return;
    double c0 = c[w * 64 + 2 * l], c1 = c[w * 64 + 2 * l + 1];
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a[w * 32 + l]), "d"(b[w * 32 + l]));
    out[w * 64 + 2 * l] = c0;
    out[w * 64 + 2 * l + 1] = c1;
}

static int reset_counter(void* ws, cudaStream_t st) {
    SMCB_CUDA(cudaMemsetAsync((char*)ws + (size_t)kRedMaxBlocks * kRedMaxVals * 8, 0, 8, st));
    return 0;
}

}  // namespace smcb

using namespace smcb;

extern "C" {

long long smcb_reduce_workspace_bytes(void) { return kRedWsBytes; }

int smcb_normals(uint64_t seed, uint32_t iteration, uint32_t stream_id, uint64_t particle0, long long N, int D,
                 double* out, void* stream) {
    SMCB_REQUIRE(out && N >= 0 && D >= 1, "bad argument");
    if (N == 0) return 0;
    normals_kernel<<<stride_grid(N * ((D + 1) / 2), 256, 8), 256, 0, (cudaStream_t)stream>>>(seed, iteration, stream_id,
                                                                                              particle0, N, D, out);
    return check_launch("normals_kernel");
}

int smcb_uniforms(uint64_t seed, uint32_t iteration, uint32_t stream_id, uint64_t particle0, long long N,
                  uint32_t draw, double* out, void* stream) {
    SMCB_REQUIRE(out && N >= 0, "bad argument");
    if (N == 0) return 0;
    uniforms_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(seed, iteration, stream_id, particle0, N,
                                                                              draw, out);
    return check_launch("uniforms_kernel");
}

static size_t tile_smem(int D) { return sizeof(double) * (size_t)kRedThreads * (D + 1); }
constexpr int kTileMaxD = 110;   // 256 rows x (D + 1) doubles must fit the 227 KB of shared memory; wider rows: one warp per row

int smcb_row_half_sqnorm(const double* r, long long N, int D, double* out, void* stream) {
    SMCB_REQUIRE(r && out && N >= 0 && D >= 1, "bad argument");
    if (N == 0) return 0;
    if (D > kTileMaxD) {
        row_sqnorm_warp_kernel<<<stride_grid(N * 32, 256, 8), 256, 0, (cudaStream_t)stream>>>(r, N, D, 0, nullptr, out);
        return check_launch("row_sqnorm_warp_kernel");
    }
    const size_t smem = tile_smem(D);
    if (smem > 48 * 1024)
        SMCB_CUDA(cudaFuncSetAttribute(row_half_sqnorm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    row_half_sqnorm_kernel<<<stride_grid(N, kRedThreads, 4), kRedThreads, smem, (cudaStream_t)stream>>>(r, N, D, out);
    return check_launch("row_half_sqnorm_kernel");
}

int smcb_std_normal_logpdf(const double* x, long long N, int D, double* out, void* stream) {
    SMCB_REQUIRE(x && out && N >= 0 && D >= 1, "bad argument");
    if (N == 0) return 0;
    if (D > kTileMaxD) {
        row_sqnorm_warp_kernel<<<stride_grid(N * 32, 256, 8), 256, 0, (cudaStream_t)stream>>>(x, N, D, 1, nullptr, out);
        return check_launch("row_sqnorm_warp_kernel");
    }
    const size_t smem = tile_smem(D);
    if (smem > 48 * 1024)
        SMCB_CUDA(cudaFuncSetAttribute(std_normal_logpdf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    std_normal_logpdf_kernel<<<stride_grid(N, kRedThreads, 4), kRedThreads, smem, (cudaStream_t)stream>>>(x, N, D, out);
    return check_launch("std_normal_logpdf_kernel");
}

int smcb_uniform_logw(const double* logZ, long long N_total, long long N, double* out, void* stream) {
    SMCB_REQUIRE(logZ && out && N >= 0 && N_total >= 1, "bad argument");
    if (N == 0) return 0;
    uniform_logw_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(logZ, log((double)N_total), N, out);
    return check_launch("uniform_logw_kernel");
}

int smcb_affine(const double* in, long long N, double a, double b, double* out, void* stream) {
    SMCB_REQUIRE(in && out && N >= 0, "bad argument");
    if (N == 0) return 0;
    affine_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(in, N, a, b, out);
    return check_launch("affine_kernel");
}

int smcb_init_logw(const double* lp, const double* x, long long N, int D, double* logw, void* stream) {
    SMCB_REQUIRE(lp && x && logw && N >= 0 && D >= 1, "bad argument");
    if (N == 0) return 0;
    if (D > kTileMaxD) {
        row_sqnorm_warp_kernel<<<stride_grid(N * 32, 256, 8), 256, 0, (cudaStream_t)stream>>>(x, N, D, 2, lp, logw);
        return check_launch("row_sqnorm_warp_kernel");
    }
    const size_t smem = tile_smem(D);
    if (smem > 48 * 1024)
        SMCB_CUDA(cudaFuncSetAttribute(init_logw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    init_logw_kernel<<<stride_grid(N, kRedThreads, 4), kRedThreads, smem, (cudaStream_t)stream>>>(lp, x, N, D, logw);
    return check_launch("init_logw_kernel");
}

int smcb_reweight_forward(const double* logw, const double* lp_x, const double* lp_xnew, const double* r,
                          const double* r_new, long long N, int D, double* out, void* stream) {
    SMCB_REQUIRE(logw && lp_x && lp_xnew && r && r_new && out && N >= 0 && D >= 1, "bad argument");
    if (N == 0) return 0;
    if (D > kTileMaxD) {
        reweight_forward_warp_kernel<<<stride_grid(N * 32, 256, 8), 256, 0, (cudaStream_t)stream>>>(logw, lp_x, lp_xnew, r,
                                                                                                   r_new, N, D, out);
        return check_launch("reweight_forward_warp_kernel");
    }
    const bool aligned = (((uintptr_t)r | (uintptr_t)r_new) % 16) == 0;
    if (aligned && (D == 4 || D == 8 || D == 16 || D == 32 || D == 64)) {
        cudaStream_t st = (cudaStream_t)stream;
        const int grid = stride_grid(N * (D / 2) / (D >= 8 ? 4 : 2), 256, 8);
        switch (D) {
            case 4: reweight_forward_coop_kernel<2><<<grid, 256, 0, st>>>(logw, lp_x, lp_xnew, r, r_new, N, out); break;
            case 8: reweight_forward_coop_kernel<4><<<grid, 256, 0, st>>>(logw, lp_x, lp_xnew, r, r_new, N, out); break;
            case 16: reweight_forward_coop_kernel<8><<<grid, 256, 0, st>>>(logw, lp_x, lp_xnew, r, r_new, N, out); break;
            case 32: reweight_forward_coop_kernel<16><<<grid, 256, 0, st>>>(logw, lp_x, lp_xnew, r, r_new, N, out); break;
            default: reweight_forward_coop_kernel<32><<<grid, 256, 0, st>>>(logw, lp_x, lp_xnew, r, r_new, N, out); break;
        }
        return check_launch("reweight_forward_coop_kernel");
    }
    const size_t smem = tile_smem(D);
    if (smem > 48 * 1024)
        SMCB_CUDA(cudaFuncSetAttribute(reweight_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    reweight_forward_kernel<<<stride_grid(N, kRedThreads, 4), kRedThreads, smem, (cudaStream_t)stream>>>(
        logw, lp_x, lp_xnew, r, r_new, N, D, out);
    return check_launch("reweight_forward_kernel");
}

int smcb_reweight_forward_split(const double* logw, const double* A_old, const double* B_old, const double* A_new,
                                const double* B_new, const double* ke_old, const double* ke_new, double phi, long long N,
                                double* out, void* stream) {
    SMCB_REQUIRE(logw && A_old && B_old && A_new && B_new && ke_old && ke_new && out && N >= 0, "bad argument");
    if (N == 0) return 0;
    reweight_forward_split_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(logw, A_old, B_old, A_new, B_new,
                                                                                         ke_old, ke_new, phi, N, out);
    return check_launch("reweight_forward_split_kernel");
}

int smcb_reweight_forward_ke(const double* logw, const double* lp_x, const double* lp_xnew, const double* ke_old,
                             const double* ke_new, long long N, double* out, void* stream) {
    SMCB_REQUIRE(logw && lp_x && lp_xnew && ke_old && ke_new && out && N >= 0, "bad argument");
    if (N == 0) return 0;
    reweight_forward_ke_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(logw, lp_x, lp_xnew, ke_old,
                                                                                         ke_new, N, out);
    return check_launch("reweight_forward_ke_kernel");
}

int smcb_reweight_general(const double* logw, const double* lp_x, const double* lp_xnew, const double* L,
                          const double* q, long long N, double* out, void* stream) {
    SMCB_REQUIRE(logw && lp_x && lp_xnew && L && q && out && N >= 0, "bad argument");
    if (N == 0) return 0;
    reweight_general_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(logw, lp_x, lp_xnew, L, q, N, out);
    return check_launch("reweight_general_kernel");
}

int smcb_reweight_asymptotic(const double* logw, const double* A, const double* B, double phi_new, double phi_old,
                             long long N, double* out, void* stream) {
    SMCB_REQUIRE(logw && A && B && out && N >= 0, "bad argument");
    if (N == 0) return 0;
    reweight_asymptotic_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(logw, A, B, phi_new, phi_old, N,
                                                                                         out);
    return check_launch("reweight_asymptotic_kernel");
}

int smcb_lse_partial(const double* logw, long long N, double* out3, void* workspace, void* stream) {
    SMCB_REQUIRE(logw && out3 && workspace && N >= 0, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (reset_counter(workspace, st)) return -1;
    lse_partial_kernel<<<stride_grid(N, kRedThreads * 8, 4), kRedThreads, 0, st>>>(logw, N, out3, (double*)workspace);
    return check_launch("lse_partial_kernel");
}

int smcb_lse_finalize(const double* triples, int P, double* out2, void* stream) {
    SMCB_REQUIRE(triples && out2 && P >= 1, "bad argument");
    lse_finalize_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(triples, P, out2);
    return check_launch("lse_finalize_kernel");
}

int smcb_normalise(const double* logw, long long N, const double* logZ, double* wn, void* stream) {
    SMCB_REQUIRE(logw && logZ && wn && N >= 0, "bad argument");
    if (N == 0) return 0;
    normalise_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(logw, N, logZ, wn);
    return check_launch("normalise_kernel");
}

int smcb_tempering_arrays(const double* A, const double* B, double phi_old, long long N, double* logpri,
                          double* loglik, double* c, void* stream) {
    SMCB_REQUIRE(A && B && logpri && loglik && c && N >= 0, "bad argument");
    if (N == 0) return 0;
    tempering_arrays_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(A, B, phi_old, N, logpri, loglik, c);
    return check_launch("tempering_arrays_kernel");
}

int smcb_ess_multi_phi(const double* loglik, const double* logpri, const double* c, long long N, const double* phis,
                       int m, double* out, void* workspace, void* stream) {
    SMCB_REQUIRE(loglik && logpri && c && phis && out && workspace && N >= 0, "bad argument");
    SMCB_REQUIRE(m >= 1 && m <= kMaxPhi, "1 <= m <= 16 candidate temperatures per pass");
    cudaStream_t st = (cudaStream_t)stream;
    if (reset_counter(workspace, st)) return -1;
    const int grid = stride_grid(N, kRedThreads * 2, 4);
    if (m == 1) ess_multi_phi_kernel<1><<<grid, kRedThreads, 0, st>>>(loglik, logpri, c, N, phis, m, out, (double*)workspace);
    else if (m <= 4) ess_multi_phi_kernel<4><<<grid, kRedThreads, 0, st>>>(loglik, logpri, c, N, phis, m, out, (double*)workspace);
    else if (m <= 8) ess_multi_phi_kernel<8><<<grid, kRedThreads, 0, st>>>(loglik, logpri, c, N, phis, m, out, (double*)workspace);
    else ess_multi_phi_kernel<16><<<grid, kRedThreads, 0, st>>>(loglik, logpri, c, N, phis, m, out, (double*)workspace);
    return check_launch("ess_multi_phi_kernel");
}

long long smcb_bisect_state_bytes(void) { return (long long)((sizeof(BisectState) + 255) / 256 * 256); }
int smcb_bisect_max_candidates(void) { return kBisectMaxCand; }
int smcb_bisect_passes(void) { return kBisectPasses; }

int smcb_bisect_init(void* state, double xa, double xb, double target, void* stream) {
    SMCB_REQUIRE(state, "bad argument");
    bisect_init_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((BisectState*)state, xa, xb, target);
    return check_launch("bisect_init_kernel");
}

int smcb_bisect_eval(const double* A, const double* B, double phi_old, long long N, const void* state, double* out,
                     void* workspace, void* stream) {
    SMCB_REQUIRE(A && B && state && out && workspace && N >= 0, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (reset_counter(workspace, st)) return -1;
    bisect_eval_kernel<<<stride_grid(N, kRedThreads * 2, 4), kRedThreads, 0, st>>>(A, B, phi_old, N, (const BisectState*)state,
                                                                                  out, (double*)workspace);
    return check_launch("bisect_eval_kernel");
}

int smcb_bisect_step(const double* triples, int P, void* state, void* stream) {
    SMCB_REQUIRE(triples && state && P >= 1, "bad argument");
    bisect_step_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(triples, P, (BisectState*)state);
    return check_launch("bisect_step_kernel");
}

int smcb_bisect_read(const void* state, double* out4, void* stream) {
    SMCB_REQUIRE(state && out4, "bad argument");
    bisect_read_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((const BisectState*)state, out4);
    return check_launch("bisect_read_kernel");
}

int smcb_weighted_moment(const double* x, const double* wn, long long N, int D, int constrain, const double* center,
                         int power, double* out, void* workspace, void* stream) {
    SMCB_REQUIRE(x && wn && out && workspace && N >= 0, "bad argument");
    SMCB_REQUIRE(D >= 1 && D <= kRedThreads && (power == 1 || power == 2), "1 <= D <= 256, power in {1, 2}");
    cudaStream_t st = (cudaStream_t)stream;
    if (reset_counter(workspace, st)) return -1;
    const int used = (kRedThreads / D) * D;
    weighted_moment_kernel<<<stride_grid(N * D, kRedThreads * 4, 4), kRedThreads, 0, st>>>(x, wn, N, D, constrain, center,
                                                                                        power, out, (double*)workspace, used);
    return check_launch("weighted_moment_kernel");
}

int smcb_scale_rows(const double* x, long long N, int D, const double* scale, int inverse, double* out, void* stream) {
    SMCB_REQUIRE(x && scale && out && N >= 0 && D >= 1, "bad argument");
    if (N == 0) return 0;
    scale_rows_kernel<<<stride_grid(N * D, 256, 8), 256, 0, (cudaStream_t)stream>>>(x, N * D, D, scale, inverse, out);
    return check_launch("scale_rows_kernel");
}

int smcb_scale_rows_accepted(const double* z, const int* accepted, const double* x, long long N, int D, const double* scale,
                             double* out, void* stream) {
    SMCB_REQUIRE(z && accepted && x && scale && out && N >= 0 && D >= 1 && out != x, "bad argument");
    if (N == 0) return 0;
    scale_rows_accepted_kernel<<<stride_grid(N * D, 256, 8), 256, 0, (cudaStream_t)stream>>>(z, accepted, x, N * D, D, scale,
                                                                                             out);
    return check_launch("scale_rows_accepted_kernel");
}

int smcb_weighted_moments12(const double* x, const double* wn, long long N, int D, int constrain, const double* center,
                            double* out2D, void* workspace, void* stream) {
    SMCB_REQUIRE(x && wn && out2D && workspace && N >= 0, "bad argument");
    SMCB_REQUIRE(D >= 1 && 2 * D <= kRedThreads, "1 <= D <= 128");
    cudaStream_t st = (cudaStream_t)stream;
    if (reset_counter(workspace, st)) return -1;
    const int used = (kRedThreads / D) * D;
    weighted_moments12_kernel<<<stride_grid(N * D, kRedThreads * 4, 4), kRedThreads, 0, st>>>(x, wn, N, D, constrain, center,
                                                                                           out2D, (double*)workspace, used);
    return check_launch("weighted_moments12_kernel");
}

int smcb_moments12_finalize(const double* sums2D, const double* center, int D, double* mean, double* var, void* stream) {
    SMCB_REQUIRE(sums2D && mean && var && D >= 1, "bad argument");
    moments12_finalize_kernel<<<(D + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sums2D, center, D, mean, var);
    return check_launch("moments12_finalize_kernel");
}

int smcb_count_moved(const double* x, const double* x_new, long long N, int D, double* out_count, void* workspace,
                     void* stream) {
    SMCB_REQUIRE(x && x_new && out_count && workspace && N >= 0 && D >= 1, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (reset_counter(workspace, st)) return -1;
    count_moved_kernel<<<stride_grid(N, kRedThreads * 2, 4), kRedThreads, 0, st>>>(x, x_new, N, D, out_count, (double*)workspace);
    return check_launch("count_moved_kernel");
}

int smcb_sum_int32(const int* v, long long N, long long* out, void* workspace, void* stream) {
    SMCB_REQUIRE(v && out && workspace && N >= 0, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (reset_counter(workspace, st)) return -1;
    sum_kernel<int, long long><<<stride_grid(N, kRedThreads * 4, 4), kRedThreads, 0, st>>>(v, N, out, (double*)workspace);
    return check_launch("sum_kernel<int>");
}

int smcb_sum_f64(const double* v, long long N, double* out, void* workspace, void* stream) {
    SMCB_REQUIRE(v && out && workspace && N >= 0, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (reset_counter(workspace, st)) return -1;
    sum_kernel<double, double><<<stride_grid(N, kRedThreads * 4, 4), kRedThreads, 0, st>>>(v, N, out, (double*)workspace);
    return check_launch("sum_kernel<double>");
}

int smcb_fast_log(const double* x, long long N, double* out, void* stream) {
    SMCB_REQUIRE(x && out && N >= 0, "bad argument");
    if (N == 0) return 0;
    fast_log_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(x, N, out);
    return check_launch("fast_log_kernel");
}

int smcb_fast_exp(const double* x, long long N, double* out, void* stream) {
    SMCB_REQUIRE(x && out && N >= 0, "bad argument");
    if (N == 0) return 0;
    fast_exp_kernel<<<stride_grid(N, 256, 8), 256, 0, (cudaStream_t)stream>>>(x, N, out);
    return check_launch("fast_exp_kernel");
}

int smcb_probe_dmma(int blocks, int threads, int iters, double* out_sink, void* stream) {
    SMCB_REQUIRE(blocks > 0 && threads > 0 && threads <= 1024 && threads % 32 == 0 && iters > 0 && out_sink, "bad argument");
    probe_dmma_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(iters, out_sink);
    return check_launch("probe_dmma_kernel");
}

int smcb_debug_dmma(const double* a, const double* b, const double* c, double* out, int nwarps, void* stream) {
    SMCB_REQUIRE(a && b && c && out && nwarps > 0, "bad argument");
    debug_dmma_kernel<<<(nwarps + 3) / 4, 128, 0, (cudaStream_t)stream>>>(a, b, c, out, nwarps);
    return check_launch("debug_dmma_kernel");
}

int smcb_probe_fp64(int blocks, int threads, int iters, double* out_sink, void* stream) {
    SMCB_REQUIRE(blocks > 0 && threads > 0 && threads <= 1024 && iters > 0 && out_sink, "bad argument");
    probe_fp64_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(iters, out_sink);
    return check_launch("probe_fp64_kernel");
}

}  // extern "C"
