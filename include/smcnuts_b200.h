/* smcnuts_b200 -- C-ABI of the B200-native SMC-NUTS particle hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / C++ types.  Every entry point
 *   - takes DEVICE pointers unless the parameter name starts with `host_`,
 *   - enqueues its work on `stream` (a cudaStream_t passed as void*) and does not synchronise,
 *   - never allocates device memory except smcb_model_create (scratch comes from the caller via the
 *     *_workspace_bytes queries), never throws,
 *   - returns 0 on success, <0 on error (message via smcb_last_error()).
 * Particle arrays are row-major [N, D] float64, exactly the reference's numpy layout.
 *
 * Each function names the reference code it replaces (paths relative to the SMC-NUTS checkout).
 * The reference has no FFI of its own for this path: its only native crossing is
 * Python -> ctypes -> BridgeStan per particle per leapfrog (smcnuts/model/bridgestan.py:46,78);
 * INTEGRATION.md shows the ctypes binding a maintainer adds to call these instead.
 */
#ifndef SMCNUTS_B200_H
#define SMCNUTS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMCB_MODEL_ARMA 0   /* stan_models/arma/arma.stan       host blob: y[T]                                   */
#define SMCB_MODEL_PRMWCD 1 /* stan_models/PRMwCD/PRMwCD.stan   host blob: q, y[NO], lgamma(y+1)[NO], X[NO*11]    */
#define SMCB_MODEL_GAUSS 2  /* synthetic Gaussian (config 4)    host blob: P[D*D] precision, row-major            */

#define SMCB_STREAM_NUTS 0
#define SMCB_STREAM_MOMENTUM 1
#define SMCB_STREAM_ACCREJ 2
#define SMCB_STREAM_RESAMPLE 3
#define SMCB_STREAM_INIT 4
#define SMCB_STREAM_ESTIMATE 5

#define SMCB_CONSTRAIN_NONE 0      /* estimate.py:34-36 (_unconstrained_target)                             */
#define SMCB_CONSTRAIN_EXP_LAST 1  /* bridgestan.py:93-120 for arma / PRMwCD: exp() on the last coordinate  */

int smcb_version(void);
/* 0: product build; 1: parity build (-DSMCB_PARITY=1 -fmad=false: the oracle's statement order in the model device
 * functions, no FMA contraction) -- libsmcnuts_b200_parity.so, loaded only by the parity tests */
int smcb_build_flavour(void);
const char* smcb_last_error(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
long long smcb_launch_count(void);

/* ---- model (replaces StanModel.__init__, bridgestan.py:13-26; phi is an argument, not a reload :122-146) */
int smcb_model_create(int kind, const double* host_data, long long n, int dim, void** handle);
/* A model that lives in its own shared object (csrc/nuts_plugin.cuh: a generated model struct compiled with the NUTS / logp
 * kernel templates).  Replaces the generic half of bridgestan.py:13-26 (any Stan program handed to BridgeStan):
 * smcnuts/model/stan_codegen.py translates a Stan program into the struct.  host_data[n] is the plug-in's data blob. */
int smcb_model_create_plugin(const char* so_path, const double* host_data, long long n, void** handle);
/* Diagonal metric of the NUTS proposal for this model: with scale[dim] set (host array; NULL restores the identity metric
 * of nuts.py:162-175), smcb_nuts_transition runs identity-metric NUTS on z = x / scale, i.e. NUTS with the mass matrix
 * diag(1 / scale^2) (README.md:66-67 "future updates").  The caller passes z and gets z back (smcb_scale_rows converts);
 * the by-products A, B stay the x-space split log density. */
int smcb_model_set_scale(void* handle, const double* host_scale);
int smcb_model_destroy(void* handle);
int smcb_model_dim(void* handle);
/* Constrained output of a plug-in model (replaces StanModel.constrain, bridgestan.py:93-120: param_constrain per particle,
 * param_num() values per row).  smcb_model_constrained_dim returns the row width CDIM (a simplex[K] has K - 1 unconstrained
 * coordinates but K values; -1 with an error for a built-in model, whose transform is fused into the moment kernels).
 * smcb_model_constrain writes out[N, CDIM] row-major (device) from the unconstrained rows x[N, dim] (device), on stream. */
int smcb_model_constrained_dim(void* handle);
int smcb_model_constrain(void* handle, const double* x, long long N, double* out, void* stream);
/* Host-only test hook (no GPU work): the tensor-core fragment packing of the PRMwCD NUTS kernel (csrc/models.cuh,
 * PrmModelG) applied to a scalar blob [16 header doubles][n_obs rows of 12]; host_out gets 32 + tiles*288 doubles. */
int smcb_debug_pack_prm(const double* host_scalar_blob, int n_obs, int tiles, double* host_out, long long n_out);

/* StanModel.logpdf / logpdfgrad (bridgestan.py:28-90): A = log prior + Jacobian, B = log likelihood,
 * grad = d(A + phi*B)/dx with the failure mapping (non-finite logp -> grad row of -inf).  Any output may be NULL. */
int smcb_logp_grad(void* handle, const double* x, long long N, double phi, double* A, double* B, double* grad,
                   void* stream);
/* out = A + phi*B, non-finite -> -inf (bridgestan.py:47-49) */
int smcb_combine_logp(const double* A, const double* B, double phi, long long N, double* out, void* stream);

/* ---- NUTS proposal (NUTSProposal.rvs nuts.py:34-175; accrej != 0: NUTSProposalWithAccRej.rvs nuts_acc_rej.py:27-52) */
int smcb_nuts_workspace_bytes(void* handle, long long N, int max_depth, long long* bytes);
/* Cap on the resident CTAs per SM of the following smcb_nuts_transition launches of the calling thread (0 = as many as
 * fit, the default).  The chunked host path of NUTSProposal.rvs (nuts.py:34-56 with host arrays) runs the launches of
 * several chunks side by side, each on a share of every SM, so that one chunk's last trees overlap the others' work. */
int smcb_nuts_set_blocks_per_sm(int blocks_per_sm);
int smcb_nuts_transition(void* handle, const double* x, const double* r, long long N, double eps, double phi,
                         int max_depth, int accrej, uint64_t seed, uint32_t iteration, uint64_t particle0,
                         double* x_new, double* r_new, double* A_old, double* B_old, double* A_new, double* B_new,
                         double* ke_old, double* ke_new, int* n_leapfrog, int* accepted, int* depth, double* accept_stat,
                         const double* A_in, const double* B_in, const double* g_in, double* g_new, void* workspace,
                         long long workspace_bytes, void* stream);
/* accept_stat (nullable): per particle, the mean over its leaves of min(1, exp(joint_leaf - joint_0)) -- the NUTS
 * acceptance statistic used by dual-averaging step-size adaptation (README.md:66-67 "future updates"; off in the
 * reference, whose step size is a run constant, nuts.py:31). */
/* A_in/B_in/g_in (all or none, accrej == 0): the split log density and gradient at x handed back from the previous
 * transition's A_new/B_new/g_new at the same phi -- the initial evaluation (nuts.py:66,72) is then skipped.
 * g_new (nullable): gradient of A + phi*B at the returned x_new. */

/* ---- Philox streams (momentum_proposal.rvs samples.py:155; sample_proposal.rvs samples.py:77) */
int smcb_normals(uint64_t seed, uint32_t iteration, uint32_t stream_id, uint64_t particle0, long long N, int D,
                 double* out, void* stream);
int smcb_uniforms(uint64_t seed, uint32_t iteration, uint32_t stream_id, uint64_t particle0, long long N,
                  uint32_t draw, double* out, void* stream);

/* ---- weights */
/* out[i] = 0.5*|r_i|^2  (momentum_proposal.logpdf(r) = -out - D/2 log 2pi, nuts.py:177-189) */
int smcb_row_half_sqnorm(const double* r, long long N, int D, double* out, void* stream);
/* out[i] = N(x_i; 0, I).logpdf = -0.5*|x_i|^2 - D/2 log 2pi  (momentum / q0 density, nuts.py:189, forward_lkernel.py:35) */
int smcb_std_normal_logpdf(const double* x, long long N, int D, double* out, void* stream);
/* out[i] = logZ[0] - log(N_total): the weights after resampling (samples.py:143) */
int smcb_uniform_logw(const double* logZ, long long N_total, long long N, double* out, void* stream);
/* out[i] = a*in[i] + b (small helper: mean = sums / N) */
int smcb_affine(const double* in, long long N, double a, double b, double* out, void* stream);
/* logw = lp - N(x; 0, I).logpdf  (samples.py:85 with q0 = N(0, I)) */
int smcb_init_logw(const double* lp, const double* x, long long N, int D, double* logw, void* stream);
/* samples.py:183-196 with ForwardLKernel (forward_lkernel.py:35): logw + lp_xnew - lp_x - 0.5|r_new|^2 + 0.5|r|^2 */
int smcb_reweight_forward(const double* logw, const double* lp_x, const double* lp_xnew, const double* r,
                          const double* r_new, long long N, int D, double* out, void* stream);
/* same, from the kinetic energies K2 already emitted (40 B/particle instead of 16D+24) */
int smcb_reweight_forward_ke(const double* logw, const double* lp_x, const double* lp_xnew, const double* ke_old,
                             const double* ke_new, long long N, double* out, void* stream);
/* the same from the split log densities emitted by smcb_nuts_transition: logp = A + phi*B (non-finite -> -inf) is formed in
 * the kernel (samples.py:190-191 evaluates logp at phi = 1 regardless of tempering: pass phi = 1) */
int smcb_reweight_forward_split(const double* logw, const double* A_old, const double* B_old, const double* A_new,
                                const double* B_new, const double* ke_old, const double* ke_new, double phi, long long N,
                                double* out, void* stream);
/* samples.py:196 for any L-kernel: logw + lp_xnew - lp_x + L - q */
int smcb_reweight_general(const double* logw, const double* lp_x, const double* lp_xnew, const double* L,
                          const double* q, long long N, double* out, void* stream);
/* samples.py:169-180: logw + logp(x, phi_new) - logp(x, phi_old) from the split at the pre-move x */
int smcb_reweight_asymptotic(const double* logw, const double* A, const double* B, double phi_new, double phi_old,
                             long long N, double* out, void* stream);

/* samples.py:96-98 + :113, pass 1: out3 = (m, sum exp(logw-m), sum exp(2(logw-m))) over finite-or-+inf entries
 * (-inf ignored).  workspace: smcb_reduce_workspace_bytes(). */
long long smcb_reduce_workspace_bytes(void);
int smcb_lse_partial(const double* logw, long long N, double* out3, void* workspace, void* stream);
/* merge P rank triples -> out2 = (logZ, ESS)   (single GPU: P = 1) */
int smcb_lse_finalize(const double* triples, int P, double* out2, void* stream);
/* samples.py:101-102: wn = exp(logw - logZ), 0 where logw = -inf; logZ read from device memory */
int smcb_normalise(const double* logw, long long N, const double* logZ, double* wn, void* stream);

/* ---- adaptive tempering (adaptive_tempering.py:18-63) */
/* logpri = A, loglik = (A+B) - A, c = A + phi_old*B, each with the -inf failure mapping (:38-39, samples.py:207) */
int smcb_tempering_arrays(const double* A, const double* B, double phi_old, long long N, double* logpri,
                          double* loglik, double* c, void* stream);
/* for each of m candidate phi: triple (max, sum exp, sum exp^2) of phi*loglik + logpri - c  (:41-54); out[m*3] */
int smcb_ess_multi_phi(const double* loglik, const double* logpri, const double* c, long long N,
                       const double* phis, int m, double* out, void* workspace, void* stream);

/* Device-resident bisection (adaptive_tempering.py:58-63: phi = 1 if ESS(1) >= alpha N else scipy.optimize.bisect(f,
 * old_phi, 1)).  The bracket, the speculative candidate temperatures of the next tree levels and the outcome live in
 * an opaque device state (smcb_bisect_state_bytes() bytes); the host enqueues init, then smcb_bisect_passes() rounds of
 * eval (+ an all-gather of the out arrays when sharded) + step, then read -- no host round trip in between; kernels
 * are no-ops once the state is final.  target = alpha * N_total.
 *   eval: out[smcb_bisect_max_candidates()][3] = (max, sum exp, sum exp^2) of phi*loglik + logpri - c per candidate,
 *         formed from the split log density (A, B) on the fly (adaptive_tempering.py:38-54)
 *   step: triples[P][max_candidates][3] in rank order -> f = ESS - target, walk, next candidates
 *   read: out4 = (phi, status, iterations, abscissa of a NaN); status 1 ok, 2 NaN value, 3 same-sign bracket, 4 no
 *         convergence (scipy's ValueError / RuntimeError cases) */
long long smcb_bisect_state_bytes(void);
int smcb_bisect_max_candidates(void);
int smcb_bisect_passes(void);
int smcb_bisect_init(void* state, double xa, double xb, double target, void* stream);
int smcb_bisect_eval(const double* A, const double* B, double phi_old, long long N, const void* state, double* out,
                     void* workspace, void* stream);
int smcb_bisect_step(const double* triples, int P, void* state, void* stream);
int smcb_bisect_read(const void* state, double* out4, void* stream);

/* ---- resampling (samples.py:116-146; `rng.choice` == searchsorted(cumsum(wn)/total, u, 'right')) */
long long smcb_scan_workspace_bytes(long long N);
/* cdf = inclusive_scan(wn) / total; total -> total_out[0].  offset_in (nullable, device) is added to every
 * prefix before normalisation and total_in (nullable) replaces the local total: the multi-GPU global scan. */
int smcb_cdf(const double* wn, long long N, const double* offset_in, const double* total_in, double* cdf,
             double* total_out, void* workspace, void* stream);
/* The same scan in two halves, the first fused with the normalisation (samples.py:101-102): wn = exp(logw - logZ) is
 * written and summed per 2048-element tile in ONE pass, the tile sums are scanned (local exclusive offsets and
 * total_out[0] stay in `workspace`); smcb_cdf_from_tilesums then writes cdf = (offset + prefix) / total, with
 * offset_total = NULL (single GPU: offset 0, local total) or a device pair (rank offset, global total) from
 * smcb_rank_offsets.  lse + normalise + scan move 8 + 16 + 16 bytes per particle in total. */
int smcb_normalise_tilesums(const double* logw, long long N, const double* logZ, double* wn, double* total_out,
                            void* workspace, void* stream);
int smcb_cdf_from_tilesums(const double* wn, long long N, const double* offset_total, double* cdf, void* workspace,
                           void* stream);
int smcb_ancestors_multinomial(const double* cdf, long long N, const double* u, long long M, int64_t* idx,
                               void* stream);
/* systematic: positions (j0 + j + u0)/M_total, j = 0..M-1 (north_star; not in the reference) */
int smcb_ancestors_systematic(const double* cdf, long long N, double u0, long long j0, long long M_total,
                              long long M, int64_t* idx, void* stream);
/* systematic ancestors + gather fused: out[j, :] = x[a_j, :], a_j = ancestor of position (j0 + j + u0)/M_total;
 * idx (nullable for D in {2,4,8,16,32,64}) receives a_j.  Replaces samples.py:139-140 in one pass. */
long long smcb_resample_workspace_bytes(long long M, int D);
/* u0_dev (nullable, device): when given, u0 is read from device memory instead (no host round trip) */
int smcb_resample_systematic(const double* cdf, long long N, double u0, const double* u0_dev, long long j0,
                             long long M_total, long long M, const double* x, int D, double* out, int64_t* idx,
                             void* workspace, void* stream);
/* Sharded variant with the particle migration FUSED into the gather: this rank serves the global output slots
 * [j0, j0+M); row j0+j is written straight into the destination rank's buffer, peer_out[(j0+j)/rows_per_rank]
 * (device array of P peer-mapped base pointers, see smcb_peer_*), over NVLink -- no send buffer, no all-to-all-v. */
int smcb_resample_systematic_push(const double* cdf, long long N, double u0, long long j0, long long M_total,
                                  long long M, const double* x, int D, double* const* peer_out, long long rows_per_rank,
                                  int64_t* idx, void* workspace, void* stream);
/* Sharded MULTINOMIAL resampling, owner-push: slot j of the global output draws u_j from Philox stream (seed, iteration,
 * stream_id, particle = j); the rank whose cdf segment holds u_j (ends[q-1] <= u_j < ends[q]; ends[P] = last cdf value of
 * every rank, all-gathered) searches its local cdf and stores the ancestor's row into peer_out[j / rows_per_rank] and the
 * global ancestor index (particle0 + local index) into peer_idx[...] (nullable).  Replaces samples.py:138-140 across
 * GPUs without gathering the cdf and without any all-to-all. */
int smcb_resample_multinomial_push(const double* cdf, long long n, const double* ends, int rank, int P, uint64_t seed,
                                   uint32_t iteration, uint32_t stream_id, long long N_total, long long particle0,
                                   const double* x, int D, double* const* peer_out, int64_t* const* peer_idx,
                                   long long rows_per_rank, void* stream);
/* out2 = (sum of totals[q] for q < rank, sum of all totals), sequential in rank order: the global-scan offsets */
int smcb_rank_offsets(const double* totals, int P, int rank, double* out2, void* stream);
/* peer-visible device buffers (CUDA IPC): alloc on the owner (64-byte handle out), open on the other ranks */
int smcb_peer_alloc(long long bytes, void** ptr, void* handle64);
int smcb_peer_open(const void* handle64, void** ptr);
int smcb_peer_close(void* ptr);
int smcb_peer_free(void* ptr);
/* out[j, :] = x[idx[j], :]  (samples.py:140) */
int smcb_gather_rows(const double* x, const int64_t* idx, long long M, int D, double* out, void* stream);

/* out[i][d] = x[i][d] * scale[d] (inverse = 0) or x[i][d] / scale[d] (inverse = 1); scale is a device array of D doubles */
int smcb_scale_rows(const double* x, long long N, int D, const double* scale, int inverse, double* out, void* stream);

/* ---- estimators (estimate.py:79-95 with constrain fused, bridgestan.py:93-120) */
/* out[d] = sum_i wn_i * (c(x_i)_d - center_d)^power ; center may be NULL (0), power in {1, 2} */
int smcb_weighted_moment(const double* x, const double* wn, long long N, int D, int constrain, const double* center,
                         int power, double* out, void* workspace, void* stream);
/* Both moments in one pass about a caller-supplied centre c (device, D doubles; NULL = 0):
 *   out2D[d] = sum_i wn_i (c(x_i)_d - c_d),  out2D[D + d] = sum_i wn_i (c(x_i)_d - c_d)^2      (D <= 128)
 * smcb_moments12_finalize turns the (all-reduced) sums into mean = c + m1 and var = m2 - m1^2 (estimate.py:91-93: the
 * same estimates; with c = the previous iteration's mean the subtraction loses nothing).  One read of x and wn and one
 * collective per SMC iteration instead of two. */
int smcb_weighted_moments12(const double* x, const double* wn, long long N, int D, int constrain, const double* center,
                            double* out2D, void* workspace, void* stream);
int smcb_moments12_finalize(const double* sums2D, const double* center, int D, double* mean, double* var, void* stream);
/* smc_sampler.py:97: number of rows with ALL coordinates changed -> out_count[0] (double) */
int smcb_count_moved(const double* x, const double* x_new, long long N, int D, double* out_count, void* workspace,
                     void* stream);

/* ---- Gaussian-approximation optimal L-kernel (gaussian_lkernel.py:24-84) */
/* sums[2D] = column sums of X = [-r_new, x_new] */
int smcb_gaussL_sums(const double* r_new, const double* x_new, long long N, int D, double* sums, void* stream);
/* gram[2D*2D] += sum_i (X_i - mean)(X_i - mean)'   (gram must be zeroed by the caller) */
int smcb_gaussL_gram(const double* r_new, const double* x_new, long long N, int D, const double* mean, double* gram,
                     void* stream);
/* cov = gram/(N_total-1) -> S = C_rr - C_rx C_xx^-1 C_xr + ridge*I = L L';  G = L^-1 [I, -C_rx C_xx^-1] (D x 2D);
 * out_logdet[2] = (log det S, path).  C_xx is inverted by Cholesky (path 0); when a pivot is not safely positive
 * (rank-deficient C_xx: N <= D+1, collapsed particles) by the pseudo-inverse with numpy's cutoff, as the reference's
 * np.linalg.pinv (gaussian_lkernel.py:64-75) (path 1); path -1: S is not positive definite, G and logdet are NaN.
 * scratch: 6*D*D doubles. */
int smcb_gaussL_factor(const double* gram, long long N_total, int D, double ridge, double* G, double* out_logdet,
                       double* scratch, void* stream);
/* out_i = -0.5*(D log 2pi + logdet + |G (X_i - mean)|^2).  scratch (nullable): smcb_gaussL_logpdf_scratch_bytes(D)
 * bytes; when given and D <= 104 the GEMM runs on the FP64 tensor cores (mma.m8n8k4). */
long long smcb_gaussL_logpdf_scratch_bytes(int D);
int smcb_gaussL_logpdf(const double* r_new, const double* x_new, long long N, int D, const double* mean,
                       const double* G, const double* logdet, double* out, double* scratch, void* stream);

/* out[0] (int64) = sum of an int32 array: the per-iteration leapfrog / grad-eval counter */
int smcb_sum_int32(const int* v, long long N, long long* out, void* workspace, void* stream);
/* out[0] = sum of a double array in fixed tile order: the summed NUTS acceptance statistic that drives the dual-averaging
 * step-size adaptation (README.md:66-67 "future updates"; the reference's step size is a run constant, nuts.py:31) */
int smcb_sum_f64(const double* v, long long N, double* out, void* workspace, void* stream);

/* out[i] = exp(x[i]) with the library's in-kernel exp (test hook: accuracy of the hot-loop exp, <= 1.5 ulp) */
int smcb_fast_exp(const double* x, long long N, double* out, void* stream);
/* test hook: the hot-loop log (csrc/common.cuh::fast_log), element-wise */
int smcb_fast_log(const double* x, long long N, double* out, void* stream);

/* test hook: one mma.m8n8k4 (FP64 tensor core) per warp on caller-supplied fragments, a[32 w], b[32 w], c[64 w] ->
 * out[64 w] (lane l holds a[l], b[l], c[2l], c[2l+1]); establishes the instruction's rounding against an exact CPU model */
int smcb_debug_dmma(const double* a, const double* b, const double* c, double* out, int nwarps, void* stream);

/* ---- measurement helper: dependent-chain-free DFMA loop; out_flops[0] = FLOPs executed (device double) */
int smcb_probe_fp64(int blocks, int threads, int iters, double* out_sink, void* stream);
/* same for the FP64 tensor-core path: 8 independent mma.m8n8k4 chains per warp, 8*512 FLOPs per warp per iteration */
int smcb_probe_dmma(int blocks, int threads, int iters, double* out_sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif
