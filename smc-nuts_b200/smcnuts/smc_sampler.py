"""SMCSampler -- the K-iteration SMC loop with a NUTS proposal (reference: smcnuts/smc_sampler.py).

Same constructor, same result attributes, same per-iteration order of operations (smc_sampler.py:109-140);
all particle state lives on the GPU.  Accepts both the constructor in the reference code
    SMCSampler(K, N, target, step_size, sample_proposal, momentum_proposal, lkernel, tempering=False, rng=...)
and the README form
    SMCSampler(K, N, target, forward_kernel, sample_proposal, tempering, lkernel, rng=...)
"""
from time import time

import numpy as np
import torch
from tqdm import tqdm

from . import _cabi, _device as dev
from .estimate.estimate import Estimate
from .estimate.estimate_from_tempered import EstimateFromTempered
from .parallel import ShardContext
from .proposal.nuts import NUTSProposal
from .proposal.nuts_acc_rej import NUTSProposalWithAccRej
from .proposal.step_size import DualAveragingStepSize
from .samples.samples import Samples


class SMCSampler:
    def __init__(self, K: int, N: int, target, step_size=None, sample_proposal=None, momentum_proposal=None,
                 lkernel="forwardsLKernel", tempering=False, rng=None, forward_kernel=None, verbose=False,
                 resampling="multinomial", save_history=None, history_budget_bytes=48 << 30, shard=None,
                 adapt_step_size=0, target_accept=0.8, adapt_mass_matrix=False):
        self.K = K  # Number of iterations
        self.N = N  # Number of particles (global)
        self.target = target
        self.rng = rng
        self.lkernel = lkernel
        self.verbose = verbose
        self.shard = shard if shard is not None else ShardContext()
        D = target.dim

        # README form: the 4th positional argument is a forward-kernel plugin, not a step size
        if forward_kernel is None and step_size is not None and hasattr(step_size, "rvs"):
            forward_kernel, step_size = step_size, None
        if forward_kernel is None:
            cls = NUTSProposalWithAccRej if lkernel == "asymptoticLKernel" else NUTSProposal  # smc_sampler.py:45-60
            forward_kernel = cls(target=self.target, momentum_proposal=momentum_proposal, step_size=step_size, rng=rng)
        self.forward_kernel = forward_kernel

        # Step-size adaptation (README.md:66-67 "future updates"; off by default = the reference's constant step size,
        # nuts.py:31): dual averaging on the NUTS acceptance statistic during the first `adapt_step_size` iterations.
        self.adapt_iters = (K // 2 if adapt_step_size is True else int(adapt_step_size or 0))
        self.adapt_iters = max(0, min(self.adapt_iters, K))
        self.step_size_adapter = None
        if self.adapt_iters:
            if not hasattr(forward_kernel, "want_accept_stat"):
                raise TypeError("adapt_step_size needs the device NUTS proposal (it emits the acceptance statistic)")
            forward_kernel.want_accept_stat = True
            self.step_size_adapter = DualAveragingStepSize(forward_kernel.step_size, target_accept)
        # Diagonal mass-matrix adaptation (same README paragraph): during the first half of the adaptation window the
        # metric follows the weighted particle variance of the unconstrained coordinates (regularised as in Stan), the
        # dual averaging restarts whenever the metric changes; both are frozen afterwards.
        self.adapt_mass_matrix = bool(adapt_mass_matrix)
        if self.adapt_mass_matrix and not (self.adapt_iters and hasattr(target, "set_metric_scale")):
            raise TypeError("adapt_mass_matrix needs adapt_step_size=K_adapt and a device model")
        self.metric_iters = self.adapt_iters // 2 if self.adapt_mass_matrix else 0
        self.metric_scale = None                # the frozen diagonal metric (host array) once adaptation has set one
        self._metric_estimator = Estimate(self.target, shard=self.shard) if self.adapt_mass_matrix else None
        self.step_sizes = np.full(K, float(getattr(forward_kernel, "step_size", np.nan)))   # step size used at iteration k
        self.accept_stat = np.full(K, np.nan)   # mean NUTS acceptance statistic of iteration k (adaptation iterations only)
        seed = getattr(forward_kernel, "seed", None)
        if seed is None:
            seed = dev.seed_from_rng(rng)
        self.seed = seed

        if lkernel == "asymptoticLKernel":
            self.estimator = EstimateFromTempered(self.target, self.N, self.K, seed, shard=self.shard,
                                                  resampling=resampling)
        else:
            self.estimator = Estimate(self.target, shard=self.shard)

        # Outputs (smc_sampler.py:66-85)
        self.resampled = [False] * (self.K + 1)
        self.ess = np.zeros(self.K + 1)
        self.log_likelihood = np.zeros(self.K + 1)
        self.phi = np.zeros(self.K + 1)
        self.acceptance_rate = np.zeros(self.K + 1)
        self.run_time = None
        self.leapfrogs = np.zeros(self.K, dtype=np.int64)   # gradient evaluations per iteration (metric counter)
        self.propose_time = np.zeros(self.K)                 # device seconds of the propose phase (CUDA events)

        self.samples = Samples(self.N, D, sample_proposal, self.target, forward_kernel, lkernel, tempering, seed,
                               resampling=resampling, shard=self.shard)
        self.samples.initialise_samples()
        n_local = self.samples.n_local

        hist_bytes = (self.K + 1) * n_local * (D + 1) * 8
        if save_history is None:
            save_history = lkernel == "asymptoticLKernel" or hist_bytes <= history_budget_bytes
        self.save_history = save_history
        if save_history:  # device-resident history (the reference keeps it in host RAM, smc_sampler.py:73-74)
            self._x_saved = dev.empty(self.K + 1, n_local, D)
            self._logw_saved = dev.empty(self.K + 1, n_local)
            self._x_saved[0].copy_(self.samples.x)
            self._logw_saved[0].copy_(self.samples.logw)
        else:
            self._x_saved = self._logw_saved = None
        self._x_saved_host = self._logw_saved_host = None

        # estimates are on the constrained scale: a simplex[K] parameter has K - 1 coordinates in x but K columns here
        DC = getattr(target, "constrained_dim", D)
        self._mean_dev = dev.zeros(self.K + 1, DC)
        self._var_dev = dev.zeros(self.K + 1, DC)
        self._moved = dev.zeros(self.K + 1)
        self.mean_estimate = np.zeros([self.K + 1, DC])
        self.variance_estimate = np.zeros([self.K + 1, DC])

    # History under the reference's names (smc_sampler.py:73-74): host NumPy arrays [K+1, N, D] / [K+1, N], materialised
    # lazily from the device-resident history on first access and cached (this rank's shard when particles are sharded).
    # `x_saved_dev` / `logw_saved_dev` are the CUDA tensors themselves.
    @property
    def x_saved(self):
        if self._x_saved is None:
            return None
        if self._x_saved_host is None:
            self._x_saved_host = self._x_saved.cpu().numpy()
        return self._x_saved_host

    @property
    def logw_saved(self):
        if self._logw_saved is None:
            return None
        if self._logw_saved_host is None:
            self._logw_saved_host = self._logw_saved.cpu().numpy()
        return self._logw_saved_host

    @property
    def x_saved_dev(self):
        return self._x_saved

    @property
    def logw_saved_dev(self):
        return self._logw_saved

    def update_sampler(self, k, mean_estimate, variance_estimate):
        """smc_sampler.py:88-97; scalars are fetched once per iteration, vectors stay on the device until the end."""
        s = self.samples
        self.log_likelihood[k] = s.log_likelihood
        self._mean_dev[k].copy_(mean_estimate)
        self._var_dev[k].copy_(variance_estimate)
        self.ess[k] = s.ess
        if s.x_new is s.x:  # after update_samples x is x_new: the reference then records 0 (smc_sampler.py:97,148)
            self._moved[k] = 0.0
        else:
            _cabi.call("smcb_count_moved", dev.ptr(s.x), dev.ptr(s.x_new), s.n_local, s.D, dev.ptr(self._moved[k:k + 1]),
                       dev.ptr(dev.reduce_ws()), dev.stream_ptr())

    def begin(self):
        """Allocate the per-run counters; sample() calls this, bench.py calls it before stepping manually."""
        self._ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(self.K)]
        self._ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(self.K)]
        self._lf = dev.zeros(self.K, dtype=torch.int64)
        self._acc_sum = dev.zeros(max(self.adapt_iters, 1))
        self._start_time = time()

    def _adapt_step_size(self, k):
        """Feed iteration k-1's mean acceptance statistic to the dual averaging and set the step size of iteration k;
        the averaged step size is frozen from iteration `adapt_iters` on."""
        if self.adapt_iters and 1 <= k <= self.adapt_iters:
            self.accept_stat[k - 1] = float(self._acc_sum[k - 1].item()) / self.N
            eps = self.step_size_adapter.update(self.accept_stat[k - 1])
            if k <= self.metric_iters:
                self._adapt_metric()
                # the step size that suited the old metric is rescaled by the geometric mean of the change and the dual
                # averaging starts over from there
                self.step_size_adapter = DualAveragingStepSize(eps * self._metric_rescale,
                                                               self.step_size_adapter.target_accept)
                eps = self.step_size_adapter.step_size
            if k == self.adapt_iters:
                eps = self.step_size_adapter.averaged()
                self.forward_kernel.want_accept_stat = False
            self.forward_kernel.step_size = eps
        if k < self.K:
            self.step_sizes[k] = self.forward_kernel.step_size

    def _adapt_metric(self):
        """scale_d = sqrt of the regularised weighted variance of unconstrained coordinate d over the current particle set
        (Stan's shrinkage: n/(n+5) var + 1e-3 * 5/(n+5) with n = ESS)."""
        s = self.samples
        _, var = self._metric_estimator.return_estimate_unconstrained(s.x, s.wn)
        var = var.cpu().numpy()
        n = max(float(s.ess), 1.0)
        var = np.where(np.isfinite(var) & (var > 0), var, 1.0)
        new = np.sqrt(n / (n + 5.0) * var + 1e-3 * 5.0 / (n + 5.0))
        old = self.target.metric_scale if self.target.metric_scale is not None else np.ones_like(new)
        self._metric_rescale = float(np.exp(np.mean(np.log(old) - np.log(new))))
        self.target.set_metric_scale(new)
        self.metric_scale = new

    def iterate(self, k):
        """One SMC iteration, in the reference's order of operations (smc_sampler.py:109-140)."""
        s = self.samples
        self.phi[k] = s.phi_new
        s.normalise_weights()
        if isinstance(self.estimator, Estimate):  # both moments in one pass about the previous iteration's mean
            mean_estimate, variance_estimate = self.estimator.return_estimate(
                s.x, s.wn, center=self._mean_dev[k - 1] if k > 0 else self._mean_dev[self.K])
        else:
            mean_estimate, variance_estimate = self.estimator.return_estimate(s.x, s.wn)
        s.prefetch_momentum()         # queued before the one host synchronisation of the iteration (ESS, below)
        s.calculate_ess()
        self._adapt_step_size(k)      # after the host synchronisation above: the previous iteration's statistic is ready
        s.resample_if_required()
        self.resampled[k] = s.resampled_last
        self._ev0[k].record()
        s.propose_samples()
        self._ev1[k].record()
        if k < self.adapt_iters:      # summed acceptance statistic of this iteration's N trees (read at iteration k + 1)
            _cabi.call("smcb_sum_f64", dev.ptr(self.forward_kernel.last["accept_stat"]), s.n_local,
                       dev.ptr(self._acc_sum[k:k + 1]), dev.ptr(dev.reduce_ws()), dev.stream_ptr())
            self.shard.all_reduce_sum_(self._acc_sum[k:k + 1])
        if getattr(s, "n_leapfrog", None) is not None:
            _cabi.call("smcb_sum_int32", dev.ptr(s.n_leapfrog), s.n_local, dev.ptr(self._lf[k:k + 1]),
                       dev.ptr(dev.reduce_ws()), dev.stream_ptr())
        s.update_temperature()
        s.reweight()
        self.update_sampler(k, mean_estimate, variance_estimate)
        s.update_samples()
        if self.save_history:
            self._x_saved[k + 1].copy_(s.x_new)
            self._logw_saved[k + 1].copy_(s.logw_new)
            self._x_saved_host = self._logw_saved_host = None

    def finish(self):
        """Final estimates from the last proposal step (smc_sampler.py:143-155)."""
        s = self.samples
        s.normalise_weights()
        mean_estimate, variance_estimate = self.estimator.return_estimate(s.x, s.wn)
        s.calculate_ess()
        self.update_sampler(self.K, mean_estimate, variance_estimate)
        self.phi[self.K] = s.phi_new

        torch.cuda.synchronize()
        self.leapfrogs = self.shard.all_reduce_sum_(self._lf.clone()).cpu().numpy()
        self.propose_time = np.array([a.elapsed_time(b) * 1e-3 for a, b in zip(self._ev0, self._ev1)])
        self.mean_estimate = self._mean_dev.cpu().numpy()
        self.variance_estimate = self._var_dev.cpu().numpy()
        self.acceptance_rate = self.shard.all_reduce_sum_(self._moved.clone()).cpu().numpy() / self.N

        # asymptotic L-kernel: re-estimate every iteration from the tempered history (smc_sampler.py:152-153)
        if self.lkernel == "asymptoticLKernel":
            self.mean_estimate, self.variance_estimate = self.estimator.estimate_from_tempered(
                self._x_saved, self._logw_saved, self.phi)

        torch.cuda.synchronize()
        self.run_time = time() - self._start_time
        if self.adapt_mass_matrix:      # the model object goes back to the identity metric; the adapted one is self.metric_scale
            self.target.set_metric_scale(None)
        s.resampler.close()           # peer-mapped migration buffers (sharded runs)
        if hasattr(self.estimator, "resampler"):
            self.estimator.resampler.close()

    def sample(self, show_progress=True):
        """Sample from the target distribution using an SMC sampler (smc_sampler.py:101-155)."""
        self.begin()
        for k in tqdm(range(self.K), desc="NUTS Sampling", disable=not show_progress):
            self.iterate(k)
        self.finish()
