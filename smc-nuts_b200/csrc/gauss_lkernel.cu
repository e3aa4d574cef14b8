// K6 -- Gaussian-approximation optimal L-kernel.
//
// Replaces /root/reference/smcnuts/lkernel/gaussian_lkernel.py:24-84, which estimates the unweighted mean
// and covariance of X = [-r_new, x_new] (N x 2D), forms the conditional Gaussian of -r_new given x_new and
// evaluates it per particle in a Python loop that recomputes pinv(C_xx) and an eigendecomposition for
// every particle (35 ms/particle at D = 100).  Here:
//   gaussL_sums    column sums (one coalesced sweep)                       -> allreduce when sharded
//   gaussL_gram    centred Gram matrix, register-tiled FP64 outer products -> allreduce when sharded
//   gaussL_factor  one CTA: Cholesky(C_xx), W = C_rx C_xx^-1, S = C_rr - W C_xr + ridge I = L L',
//                  G = L^-1 [I, -W], log det S
//   gaussL_logpdf  per particle: z = G (X_i - mean), -0.5 (D log 2pi + log det S + |z|^2)
// which is algebraically the reference's multivariate_normal.logpdf(-r_i; mu_i, S) with
// mu_i = mu_r + W (x_i - mu_x)  (hoisted form checked to ~1e-13 against the reference loop in tests/golden).
#include "capi.cuh"

namespace smcb {

// X_ic for the virtual matrix X = [-r_new, x_new]
__device__ __forceinline__ double xval(const double* __restrict__ r, const double* __restrict__ x, long long i, int c,
                                       int D) {
    return (c < D) ? -r[i * D + c] : x[i * D + (c - D)];
}

__global__ void __launch_bounds__(256) gaussL_sums_kernel(const double* __restrict__ r, const double* __restrict__ x,
                                                          long long N, int D, double* sums, int used) {
    __shared__ double sh[256];
    const long long total = N * D;
    const long long gstride = (long long)gridDim.x * used;
    const int col = threadIdx.x % D;
    double ar = 0.0, ax = 0.0;
    if ((int)threadIdx.x < used)
        for (long long e = (long long)blockIdx.x * used + threadIdx.x; e < total; e += gstride) {
            ar -= r[e];
            ax += x[e];
        }
    for (int pass = 0; pass < 2; ++pass) {
        sh[threadIdx.x] = pass ? ax : ar;
        __syncthreads();
        if ((int)threadIdx.x < D) {
            double s = 0.0;
            for (int t = threadIdx.x; t < used; t += D) s += sh[t];
            atomicAdd(&sums[pass * D + col], s);
        }
        __syncthreads();
    }
}

// Centred Gram: each CTA owns one TB x TB output tile and a slab of rows; 16 x 16 threads, 4 x 4 micro-tiles.
constexpr int kTB = 64, kTM = 4, kRK = 32;
__global__ void __launch_bounds__(256) gaussL_gram_kernel(const double* __restrict__ r, const double* __restrict__ x,
                                                          long long N, int D, const double* __restrict__ mean,
                                                          double* gram, int tiles, long long rows_per_block) {
    __shared__ double smA[kRK][kTB + 2], smB[kRK][kTB + 2];
    const int D2 = 2 * D;
    const int ti = blockIdx.y / tiles, tj = blockIdx.y % tiles;
    if (tj < ti) return;  // symmetric: only the upper block-triangle is accumulated, mirrored in gaussL_factor
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const long long row_begin = (long long)blockIdx.x * rows_per_block;
    const long long row_end = min(N, row_begin + rows_per_block);
    double acc[kTM][kTM];
#pragma unroll
    for (int a = 0; a < kTM; ++a)
#pragma unroll
        for (int b = 0; b < kTM; ++b) acc[a][b] = 0.0;
    for (long long row0 = row_begin; row0 < row_end; row0 += kRK) {
        for (int e = threadIdx.x; e < kRK * kTB; e += 256) {
            const int k = e / kTB, c = e % kTB;
            const long long i = row0 + k;
            const int ca = ti * kTB + c, cb = tj * kTB + c;
            smA[k][c] = (i < row_end && ca < D2) ? xval(r, x, i, ca, D) - mean[ca] : 0.0;
            smB[k][c] = (i < row_end && cb < D2) ? xval(r, x, i, cb, D) - mean[cb] : 0.0;
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < kRK; ++k) {
            double a[kTM], b[kTM];
#pragma unroll
            for (int m = 0; m < kTM; ++m) { a[m] = smA[k][ty * kTM + m]; b[m] = smB[k][tx * kTM + m]; }
#pragma unroll
            for (int m = 0; m < kTM; ++m)
#pragma unroll
                for (int n = 0; n < kTM; ++n) acc[m][n] += a[m] * b[n];
        }
        __syncthreads();
    }
#pragma unroll
    for (int m = 0; m < kTM; ++m)
#pragma unroll
        for (int n = 0; n < kTM; ++n) {
            const int gi = ti * kTB + ty * kTM + m, gj = tj * kTB + tx * kTM + n;
            if (gi < D2 && gj < D2) atomicAdd(&gram[(size_t)gi * D2 + gj], acc[m][n]);
        }
}

// ------------------------------------------------------------------------------------------ FP64 tensor-core path
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// Centred Gram with mma.m8n8k4 (k = particles): a CTA stages 32 centred rows x C8*8 columns in shared memory; each of
// its 8 warps owns one 32 x 32 output block (pair of 4-tile column groups, upper triangle only) and accumulates it in
// 16 tile accumulators over the whole row slab; one atomicAdd per output element per CTA at the end.
constexpr int kGramRows = 32;
__global__ void __launch_bounds__(256) gaussL_gram_dmma_kernel(const double* __restrict__ r, const double* __restrict__ x,
                                                               long long N, int D, const double* __restrict__ mean,
                                                               double* gram, int C8, int nblk, int npairs,
                                                               long long rows_per_block) {
    extern __shared__ double sm[];  // [kGramRows][ld]
    const int D2 = 2 * D, W = C8 * 8, ld = W + 4;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int pair = blockIdx.y * 8 + warp;
    // decode pair -> (bi <= bj) over nblk column blocks of 32
    int bi = 0, bj = 0;
    {
        int t = pair, row = 0;
        while (row < nblk && t >= nblk - row) { t -= nblk - row; ++row; }
        bi = row; bj = row + t;
    }
    const bool active = pair < npairs;
    double acc[4][4][2];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
    const long long row_begin = (long long)blockIdx.x * rows_per_block;
    const long long row_end = min(N, row_begin + rows_per_block);
    for (long long row0 = row_begin; row0 < row_end; row0 += kGramRows) {
        for (int e = threadIdx.x; e < kGramRows * W; e += 256) {
            const int k = e / W, c = e - k * W;
            const long long i = row0 + k;
            sm[k * ld + c] = (i < row_end && c < D2) ? xval(r, x, i, c, D) - mean[c] : 0.0;
        }
        __syncthreads();
        if (active) {
#pragma unroll
            for (int kk = 0; kk < kGramRows / 4; ++kk) {
                const double* rowp = sm + (4 * kk + (lane & 3)) * ld + (lane >> 2);
                double av[4], bv[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const int ca = bi * 32 + 8 * t, cb = bj * 32 + 8 * t;
                    av[t] = ca < W ? rowp[ca] : 0.0;
                    bv[t] = cb < W ? rowp[cb] : 0.0;
                }
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b) dmma884(acc[a][b][0], acc[a][b][1], av[a], bv[b]);
            }
        }
        __syncthreads();
    }
    if (active) {
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int gi = bi * 32 + 8 * a + (lane >> 2), gj = bj * 32 + 8 * b + 2 * (lane & 3) + e;
                    if (gi < D2 && gj < D2 && gi <= gj) atomicAdd(&gram[(size_t)gi * D2 + gj], acc[a][b][e]);
                }
    }
}

// B-fragment packing of G' for the logpdf GEMM: frag[(nt*KK + kk)*32 + l] = G[8nt + l/4][4kk + l%4] (0 outside)
__global__ void gaussL_pack_G_kernel(const double* __restrict__ G, int D, int NT8, int KK, double* __restrict__ frag) {
    const int total = NT8 * KK * 32;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
        const int l = t & 31, kk = (t >> 5) % KK, nt = (t >> 5) / KK;
        const int n = 8 * nt + (l >> 2), k = 4 * kk + (l & 3);
        frag[t] = (n < D && k < 2 * D) ? G[(size_t)n * 2 * D + k] : 0.0;
    }
}

// z = G (X_i - mean) for 8 particles per warp (4 lanes per particle), |z|^2 folded in the group.
template <int NT8>
__global__ void __launch_bounds__(256) gaussL_logpdf_dmma_kernel(const double* __restrict__ r, const double* __restrict__ x,
                                                                 long long N, int D, const double* __restrict__ mean,
                                                                 const double* __restrict__ frag, int KK,
                                                                 const double* __restrict__ logdet,
                                                                 double* __restrict__ out) {
    extern __shared__ double sm[];  // frag [NT8][KK][32]
    for (int t = threadIdx.x; t < NT8 * KK * 32; t += blockDim.x) sm[t] = frag[t];
    __syncthreads();
    const int lane = threadIdx.x & 31, sub = lane & 3, D2 = 2 * D;
    const double c0 = D * kLog2Pi + logdet[0];
    const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    const long long wid = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (long long p0 = wid * 8; p0 < N; p0 += nwarps * 8) {
        const long long i = p0 + (lane >> 2);
        const bool ok = i < N;
        double c[2 * NT8];
#pragma unroll
        for (int j = 0; j < 2 * NT8; ++j) c[j] = 0.0;
        for (int kk = 0; kk < KK; ++kk) {
            const int k = 4 * kk + sub;
            const double av = (ok && k < D2) ? xval(r, x, i, k, D) - mean[k] : 0.0;
            const double* bp = sm + (size_t)kk * 32 + lane;
#pragma unroll
            for (int nt = 0; nt < NT8; ++nt) dmma884(c[2 * nt], c[2 * nt + 1], av, bp[(size_t)nt * KK * 32]);
        }
        double maha = 0.0;
#pragma unroll
        for (int j = 0; j < 2 * NT8; ++j) maha += c[j] * c[j];
        maha += __shfl_xor_sync(0xffffffffu, maha, 1);
        maha += __shfl_xor_sync(0xffffffffu, maha, 2);
        if (ok && sub == 0) out[i] = -0.5 * (c0 + maha);
    }
}

// In-place lower Cholesky of the n x n row-major matrix a (only the lower triangle is read).  One CTA.
// A pivot that is not safely positive (<= tol, or NaN) sets *fail and stops: the caller then takes the pseudo-inverse
// path (a rank-deficient C_xx: N <= D + 1, or particles collapsed onto few distinct rows after resampling -- the
// reference inverts with np.linalg.pinv, gaussian_lkernel.py:64-75, and stays finite there).
__device__ void chol_inplace(double* a, int n, double tol, int* fail) {
    for (int j = 0; j < n; ++j) {
        __syncthreads();
        if (threadIdx.x == 0) {
            const double d = a[j * n + j];
            if (!(d > tol)) *fail = 1;
            a[j * n + j] = sqrt(d);
        }
        __syncthreads();
        if (*fail) return;
        const double dj = a[j * n + j];
        for (int i = j + 1 + threadIdx.x; i < n; i += blockDim.x) a[i * n + j] /= dj;
        __syncthreads();
        // trailing update of the lower triangle
        const int rem = n - j - 1;
        for (int t = threadIdx.x; t < rem * rem; t += blockDim.x) {
            const int i = j + 1 + t / rem, k = j + 1 + t % rem;
            if (k <= i) a[i * n + k] -= a[i * n + j] * a[k * n + j];
        }
    }
    __syncthreads();
}

// Moore-Penrose pseudo-inverse of the symmetric n x n matrix A (full storage, destroyed) by cyclic Jacobi with a
// round-robin parallel ordering: every round rotates n/2 disjoint (p, q) pairs at once.  pinv = sum over
// |lambda_i| > rcond * max|lambda| of v_i v_i' / lambda_i with rcond = 1e-15, numpy.linalg.pinv's default cutoff
// (for a symmetric matrix the singular values are |lambda_i|).  One CTA; V and out are n x n scratch / result.
__device__ void pinv_sym_jacobi(double* A, double* V, double* out, int n) {
    __shared__ double rot_c[64], rot_s[64];
    __shared__ int rot_p[64], rot_q[64];
    __shared__ double lam_max, scale0;
    __shared__ int active;
    for (int t = threadIdx.x; t < n * n; t += blockDim.x) V[t] = (t / n == t % n) ? 1.0 : 0.0;
    if (threadIdx.x == 0) {
        double mx = 0.0;
        for (int i = 0; i < n; ++i) mx = fmax(mx, fabs(A[i * n + i]));
        scale0 = mx;
    }
    __syncthreads();
    const int ne = (n + 1) & ~1, m = ne - 1, npairs = ne / 2;   // ne players (index n = bye when n is odd)
    for (int sweep = 0; sweep < 30; ++sweep) {
        if (threadIdx.x == 0) active = 0;
        __syncthreads();
        for (int r = 0; r < m; ++r) {
            if ((int)threadIdx.x < npairs) {
                const int k = threadIdx.x;
                int pp = (k == 0) ? m : (r + k) % m;
                int qq = (k == 0) ? r % m : (r - k + m) % m;
                if (pp > qq) { const int t_ = pp; pp = qq; qq = t_; }
                double c = 1.0, sn = 0.0;
                if (qq < n) {
                    const double apq = A[pp * n + qq], app = A[pp * n + pp], aqq = A[qq * n + qq];
                    // rotate while the off-diagonal entry matters relative to its diagonal pair and to the matrix scale
                    if (fabs(apq) > 1e-22 * scale0 && fabs(apq) > 1e-17 * sqrt(fabs(app * aqq))) {
                        const double tau = (aqq - app) / (2.0 * apq);
                        const double tt = (tau >= 0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
                        c = rsqrt(1.0 + tt * tt);
                        sn = tt * c;
                        active = 1;
                    }
                } else {
                    qq = pp;   // bye
                }
                rot_p[k] = pp; rot_q[k] = qq; rot_c[k] = c; rot_s[k] = sn;
            }
            __syncthreads();
            // rows:  A <- J' A
            for (int t = threadIdx.x; t < npairs * n; t += blockDim.x) {
                const int k = t / n, j = t % n, pp = rot_p[k], qq = rot_q[k];
                if (pp == qq) continue;
                const double c = rot_c[k], sn = rot_s[k], x = A[pp * n + j], y = A[qq * n + j];
                A[pp * n + j] = c * x - sn * y;
                A[qq * n + j] = sn * x + c * y;
            }
            __syncthreads();
            // columns:  A <- A J,  V <- V J
            for (int t = threadIdx.x; t < npairs * n; t += blockDim.x) {
                const int k = t / n, i = t % n, pp = rot_p[k], qq = rot_q[k];
                if (pp == qq) continue;
                const double c = rot_c[k], sn = rot_s[k];
                double x = A[i * n + pp], y = A[i * n + qq];
                A[i * n + pp] = c * x - sn * y;
                A[i * n + qq] = sn * x + c * y;
                x = V[i * n + pp]; y = V[i * n + qq];
                V[i * n + pp] = c * x - sn * y;
                V[i * n + qq] = sn * x + c * y;
            }
            __syncthreads();
        }
        if (!active) break;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double mx = 0.0;
        for (int i = 0; i < n; ++i) mx = fmax(mx, fabs(A[i * n + i]));
        lam_max = mx;
    }
    __syncthreads();
    const double cutoff = 1e-15 * lam_max;
    for (int t = threadIdx.x; t < n * n; t += blockDim.x) {
        const int i = t / n, j = t % n;
        double acc = 0.0;
        for (int k = 0; k < n; ++k) {
            const double lam = A[k * n + k];
            if (fabs(lam) > cutoff) acc += V[i * n + k] * V[j * n + k] / lam;
        }
        out[t] = acc;
    }
    __syncthreads();
}

// Solve L Y = B in place (B is n x m row-major, L lower-triangular n x n).  One thread per column of B.
__device__ void trsm_lower(const double* L, double* B, int n, int m) {
    for (int c = threadIdx.x; c < m; c += blockDim.x)
        for (int i = 0; i < n; ++i) {
            double s = B[i * m + c];
            for (int k = 0; k < i; ++k) s -= L[i * n + k] * B[k * m + c];
            B[i * m + c] = s / L[i * n + i];
        }
    __syncthreads();
}
// Solve L' Y = B in place.
__device__ void trsm_lower_t(const double* L, double* B, int n, int m) {
    for (int c = threadIdx.x; c < m; c += blockDim.x)
        for (int i = n - 1; i >= 0; --i) {
            double s = B[i * m + c];
            for (int k = i + 1; k < n; ++k) s -= L[k * n + i] * B[k * m + c];
            B[i * m + c] = s / L[i * n + i];
        }
    __syncthreads();
}

__global__ void __launch_bounds__(256) gaussL_factor_kernel(const double* __restrict__ gram, long long N_total, int D,
                                                            double ridge, double* G, double* out_logdet,
                                                            double* scratch) {
    __shared__ int fail;
    __shared__ double scale;
    const int D2 = 2 * D, DD = D * D;
    double* Lx = scratch;           // C_xx -> chol
    double* Wt = scratch + DD;      // C_xr (D x D) -> C_xx^-1 C_xr = W'
    double* S = scratch + 2 * DD;   // S -> chol
    const double inv = 1.0 / (double)(N_total - 1);  // np.cov ddof = 1 (gaussian_lkernel.py:49)
    auto cov = [&](int i, int j) { return (i <= j ? gram[(size_t)i * D2 + j] : gram[(size_t)j * D2 + i]) * inv; };
    for (int t = threadIdx.x; t < DD; t += blockDim.x) {
        const int i = t / D, j = t % D;
        Lx[t] = cov(D + i, D + j);
        Wt[t] = cov(D + i, j);  // C_xr[i][j]
    }
    if (threadIdx.x == 0) {
        fail = 0;
        double mx = 0.0;
        for (int i = 0; i < D; ++i) mx = fmax(mx, cov(D + i, D + i));
        scale = mx;
    }
    __syncthreads();
    int path = 0;
    chol_inplace(Lx, D, 1e-13 * scale, &fail);
    __syncthreads();
    if (!fail) {
        trsm_lower(Lx, Wt, D, D);
        trsm_lower_t(Lx, Wt, D, D);  // Wt = C_xx^-1 C_xr, i.e. W = Wt'
    } else {
        // rank-deficient / indefinite C_xx: W' = pinv(C_xx) C_xr as the reference (gaussian_lkernel.py:64-75)
        path = 1;
        double* Afull = scratch + 3 * DD;
        double* V = scratch + 4 * DD;
        double* Pinv = scratch + 5 * DD;
        for (int t = threadIdx.x; t < DD; t += blockDim.x) Afull[t] = cov(D + t / D, D + t % D);
        __syncthreads();
        pinv_sym_jacobi(Afull, V, Pinv, D);
        for (int t = threadIdx.x; t < DD; t += blockDim.x) {
            const int i = t / D, j = t % D;
            double acc = 0.0;
            for (int k = 0; k < D; ++k) acc += Pinv[i * D + k] * cov(D + k, j);
            Wt[t] = acc;
        }
        __syncthreads();
        if (threadIdx.x == 0) fail = 0;
        __syncthreads();
    }
    for (int t = threadIdx.x; t < DD; t += blockDim.x) {
        const int i = t / D, j = t % D;
        double s = cov(i, j);
        for (int k = 0; k < D; ++k) s -= cov(i, D + k) * Wt[k * D + j];  // C_rx[i][k] * (C_xx^-1 C_xr)[k][j]
        S[t] = s + (i == j ? ridge : 0.0);
    }
    __syncthreads();
    // symmetrise the lower triangle that the factorisation reads
    for (int t = threadIdx.x; t < DD; t += blockDim.x) {
        const int i = t / D, j = t % D;
        if (j < i) S[t] = 0.5 * (S[t] + S[j * D + i]);
    }
    __syncthreads();
    chol_inplace(S, D, 0.0, &fail);
    __syncthreads();
    if (threadIdx.x == 0) {
        double ld = 0.0;
        for (int i = 0; i < D; ++i) ld += log(S[i * D + i]);
        out_logdet[0] = fail ? __longlong_as_double(0x7ff8000000000000LL) : 2.0 * ld;
        out_logdet[1] = fail ? -1.0 : (double)path;   // 0: Cholesky of C_xx, 1: pseudo-inverse path, -1: S not positive definite
    }
    if (fail) {   // poison G so that the failure cannot pass silently as finite weights
        for (int t = threadIdx.x; t < D * D2; t += blockDim.x) G[t] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    // G = L^-1 [I, -W]   (D x 2D)
    for (int t = threadIdx.x; t < D * D2; t += blockDim.x) {
        const int i = t / D2, c = t % D2;
        G[t] = (c < D) ? (i == c ? 1.0 : 0.0) : -Wt[(c - D) * D + i];  // -W[i][c-D] = -Wt[c-D][i]
    }
    __syncthreads();
    trsm_lower(S, G, D, D2);
}

constexpr int kGDmax = 128;
__global__ void __launch_bounds__(128) gaussL_logpdf_kernel(const double* __restrict__ r, const double* __restrict__ x,
                                                            long long N, int D, const double* __restrict__ mean,
                                                            const double* __restrict__ G,
                                                            const double* __restrict__ logdet, double* __restrict__ out,
                                                            int g_in_smem) {
    extern __shared__ double sm[];
    const int D2 = 2 * D;
    const double* Gs = G;
    if (g_in_smem) {
        for (int t = threadIdx.x; t < D * D2; t += blockDim.x) sm[t] = G[t];
        __syncthreads();
        Gs = sm;
    }
    const double c0 = D * kLog2Pi + logdet[0];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
        double v[2 * kGDmax];
        for (int c = 0; c < D2; ++c) v[c] = xval(r, x, i, c, D) - mean[c];
        double maha = 0.0;
        for (int row = 0; row < D; ++row) {
            const double* g = Gs + (size_t)row * D2;
            double z = 0.0;
#pragma unroll 4
            for (int c = 0; c < D2; ++c) z += g[c] * v[c];
            maha += z * z;
        }
        out[i] = -0.5 * (c0 + maha);
    }
}

}  // namespace smcb

using namespace smcb;

extern "C" {

int smcb_gaussL_sums(const double* r_new, const double* x_new, long long N, int D, double* sums, void* stream) {
    SMCB_REQUIRE(r_new && x_new && sums && N >= 1 && D >= 1 && D <= kGDmax, "bad argument (D <= 128)");
    cudaStream_t st = (cudaStream_t)stream;
    SMCB_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * 2 * D, st));
    const int used = (256 / D) * D;
    gaussL_sums_kernel<<<stride_grid(N * D, 256, 4), 256, 0, st>>>(r_new, x_new, N, D, sums, used);
    return check_launch("gaussL_sums_kernel");
}

int smcb_gaussL_gram(const double* r_new, const double* x_new, long long N, int D, const double* mean, double* gram,
                     void* stream) {
    SMCB_REQUIRE(r_new && x_new && mean && gram && N >= 1 && D >= 1 && D <= kGDmax, "bad argument (D <= 128)");
    if (D <= 104) {   // FP64 tensor-core path
        const int C8 = (2 * D + 7) / 8, W = C8 * 8, nblk = (W + 31) / 32, npairs = nblk * (nblk + 1) / 2;
        const int gy = (npairs + 7) / 8;
        long long slabs = (long long)device_sm_count() * 2 / gy;
        if (slabs < 1) slabs = 1;
        long long rpb = (N + slabs - 1) / slabs;
        rpb = ((rpb + kGramRows - 1) / kGramRows) * kGramRows;
        slabs = (N + rpb - 1) / rpb;
        const size_t smem = sizeof(double) * (size_t)kGramRows * (W + 4);
        if (smem > 48 * 1024)
            SMCB_CUDA(cudaFuncSetAttribute(gaussL_gram_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        dim3 grid((unsigned)slabs, (unsigned)gy);
        gaussL_gram_dmma_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(r_new, x_new, N, D, mean, gram, C8, nblk, npairs, rpb);
        return check_launch("gaussL_gram_dmma_kernel");
    }
    const int tiles = (2 * D + kTB - 1) / kTB;
    const int active_tiles = tiles * (tiles + 1) / 2;
    long long slabs = (long long)device_sm_count() * 4 / active_tiles;
    if (slabs < 1) slabs = 1;
    long long rows_per_block = (N + slabs - 1) / slabs;
    rows_per_block = ((rows_per_block + kRK - 1) / kRK) * kRK;
    slabs = (N + rows_per_block - 1) / rows_per_block;
    dim3 grid((unsigned)slabs, (unsigned)(tiles * tiles));
    gaussL_gram_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(r_new, x_new, N, D, mean, gram, tiles, rows_per_block);
    return check_launch("gaussL_gram_kernel");
}

int smcb_gaussL_factor(const double* gram, long long N_total, int D, double ridge, double* G, double* out_logdet,
                       double* scratch, void* stream) {
    SMCB_REQUIRE(gram && G && out_logdet && scratch && N_total >= 2 && D >= 1 && D <= kGDmax, "bad argument (D <= 128)");
    gaussL_factor_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(gram, N_total, D, ridge, G, out_logdet, scratch);
    return check_launch("gaussL_factor_kernel");
}

// FP64 tensor-core logpdf (D <= 104): NT8 n-tiles of 8 rows of G, KK k-steps of 4 columns; the packed fragments of G'
// take NT8 * KK * 32 doubles of the caller's scratch
static int gaussL_nt8(int D) { return D <= 8 ? 1 : D <= 16 ? 2 : D <= 32 ? 4 : D <= 64 ? 8 : 13; }
static int gaussL_kk(int D) { return (2 * D + 3) / 4; }

long long smcb_gaussL_logpdf_scratch_bytes(int D) {
    if (D < 1 || D > 104) return 0;   // scalar path: no scratch
    return (long long)sizeof(double) * gaussL_nt8(D) * gaussL_kk(D) * 32;
}

int smcb_gaussL_logpdf(const double* r_new, const double* x_new, long long N, int D, const double* mean,
                       const double* G, const double* logdet, double* out, double* scratch, void* stream) {
    SMCB_REQUIRE(r_new && x_new && mean && G && logdet && out && N >= 0 && D >= 1 && D <= kGDmax, "bad argument (D <= 128)");
    if (N == 0) return 0;
    if (D <= 104 && scratch) {   // FP64 tensor-core path; scratch holds the packed fragments of G'
        cudaStream_t st = (cudaStream_t)stream;
        const int NT8 = gaussL_nt8(D);
        const int KK = gaussL_kk(D);
        const int nfrag = NT8 * KK * 32;
        gaussL_pack_G_kernel<<<(nfrag + 255) / 256, 256, 0, st>>>(G, D, NT8, KK, scratch);
        if (check_launch("gaussL_pack_G_kernel")) return -1;
        const size_t smem = sizeof(double) * (size_t)nfrag;
        const int grid = stride_grid((N + 7) / 8 * 32, 256, smem > 100 * 1024 ? 1 : 2);
#define LAUNCH_LP(K)                                                                                                          \
    do {                                                                                                                      \
        if (smem > 48 * 1024)                                                                                                 \
            SMCB_CUDA(cudaFuncSetAttribute(gaussL_logpdf_dmma_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        gaussL_logpdf_dmma_kernel<K><<<grid, 256, smem, st>>>(r_new, x_new, N, D, mean, scratch, KK, logdet, out);              \
    } while (0)
        switch (NT8) {
            case 1: LAUNCH_LP(1); break;
            case 2: LAUNCH_LP(2); break;
            case 4: LAUNCH_LP(4); break;
            case 8: LAUNCH_LP(8); break;
            default: LAUNCH_LP(13); break;
        }
#undef LAUNCH_LP
        return check_launch("gaussL_logpdf_dmma_kernel");
    }
    const size_t smem = sizeof(double) * (size_t)D * 2 * D;
    const int in_smem = smem <= 200 * 1024;
    if (in_smem && smem > 48 * 1024)
        SMCB_CUDA(cudaFuncSetAttribute(gaussL_logpdf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gaussL_logpdf_kernel<<<stride_grid(N, 128, in_smem && smem > 100 * 1024 ? 1 : 4), 128, in_smem ? smem : 0,
                           (cudaStream_t)stream>>>(r_new, x_new, N, D, mean, G, logdet, out, in_smem);
    return check_launch("gaussL_logpdf_kernel");
}

}  // extern "C"
